"""Artefact formats of the FPL+ recipe on the host (SURVEY.md section 8 f-4): NIfTI-1 volumes without SimpleITK,
the ``image,label,pixel_weight,image_weight`` training CSV, the image-weight table derived from the sorted
uncertainties (the reference's missing ``data/get image_weight.py``, README.md:74), pixel-weight volumes, and the
Dice / ASSD evaluation.  Plain numpy / scipy: this is file I/O around the hot path, not part of it.

References: PyMIC/pymic/io/image_read_write.py:9-37 (load_nifty_volume_as_4d_array), :92-108
(save_array_as_nifty_volume), :69-90 / :130-148 (format dispatch); data/get_pixel_weight.py:12-28;
PyMIC/pymic/util/evaluation_seg_train.py:21-50 (binary_dice), :83-99 (get_edge_points), :139-172 (binary_assd);
config_dual/data_vs/train_vs_t1s_wi+wp.csv (CSV layout); net_run_dsbn/agent_seg.py:954-960 (sorted .npy layout).
"""
import csv
import gzip
import os
import struct

import numpy as np

# NIfTI-1 datatype codes <-> numpy
_NIFTI_DTYPES = {2: np.uint8, 4: np.int16, 8: np.int32, 16: np.float32, 64: np.float64, 256: np.int8, 512: np.uint16,
                 768: np.uint32, 1024: np.int64, 1280: np.uint64}
_NIFTI_CODES = {np.dtype(v): k for k, v in _NIFTI_DTYPES.items()}


def _quat_to_rot(b, c, d):
    a = np.sqrt(max(0.0, 1.0 - (b * b + c * c + d * d)))
    return np.array([[a * a + b * b - c * c - d * d, 2 * (b * c - a * d), 2 * (b * d + a * c)],
                     [2 * (b * c + a * d), a * a + c * c - b * b - d * d, 2 * (c * d - a * b)],
                     [2 * (b * d - a * c), 2 * (c * d + a * b), a * a + d * d - b * b - c * c]])


def _rot_to_quat(r):
    """Rotation matrix (det +1) -> (b, c, d) of the NIfTI quaternion with a >= 0."""
    tr = r[0, 0] + r[1, 1] + r[2, 2]
    if tr > 0:
        a = 0.5 * np.sqrt(1.0 + tr)
        b, c, d = (r[2, 1] - r[1, 2]) / (4 * a), (r[0, 2] - r[2, 0]) / (4 * a), (r[1, 0] - r[0, 1]) / (4 * a)
    else:
        i = int(np.argmax([r[0, 0], r[1, 1], r[2, 2]]))
        j, k = (i + 1) % 3, (i + 2) % 3
        q = [0.0, 0.0, 0.0]
        q[i] = 0.5 * np.sqrt(max(0.0, 1.0 + r[i, i] - r[j, j] - r[k, k]))
        a = (r[k, j] - r[j, k]) / (4 * q[i])
        q[j], q[k] = (r[j, i] + r[i, j]) / (4 * q[i]), (r[k, i] + r[i, k]) / (4 * q[i])
        b, c, d = q
        if a < 0:
            b, c, d = -b, -c, -d
    return float(b), float(c), float(d)


def read_nifti(filename):
    """Single-file NIfTI-1 (.nii / .nii.gz) -> dict(data [z,y,x] or [t,z,y,x], spacing (x,y,z), origin (x,y,z) and
    direction (9 floats, row major) in ITK's LPS convention -- what SimpleITK's ReadImage / GetArrayFromImage return."""
    opener = gzip.open if str(filename).endswith(".gz") else open
    with opener(filename, "rb") as f:
        raw = f.read()
    if len(raw) < 352:
        raise ValueError("%s: not a NIfTI-1 file" % filename)
    endian = "<" if struct.unpack("<i", raw[:4])[0] == 348 else ">"
    if struct.unpack(endian + "i", raw[:4])[0] != 348:
        raise ValueError("%s: sizeof_hdr != 348" % filename)
    if raw[344:348] not in (b"n+1\0", b"ni1\0"):
        raise ValueError("%s: bad NIfTI magic %r" % (filename, raw[344:348]))
    if raw[344:348] == b"ni1\0":
        raise ValueError("%s: two-file NIfTI (.hdr/.img) is not supported" % filename)
    dim = struct.unpack(endian + "8h", raw[40:56])
    datatype, = struct.unpack(endian + "h", raw[70:72])
    pixdim = struct.unpack(endian + "8f", raw[76:108])
    vox_offset, scl_slope, scl_inter = struct.unpack(endian + "3f", raw[108:120])
    qform_code, sform_code = struct.unpack(endian + "2h", raw[252:256])
    quatern = struct.unpack(endian + "3f", raw[256:268])
    qoffset = struct.unpack(endian + "3f", raw[268:280])
    srow = np.array(struct.unpack(endian + "12f", raw[280:328]), np.float64).reshape(3, 4)
    if datatype not in _NIFTI_DTYPES:
        raise ValueError("%s: unsupported NIfTI datatype %d" % (filename, datatype))
    ndim = dim[0]
    shape = [int(d) for d in dim[1:1 + ndim]]
    while len(shape) > 3 and shape[-1] == 1:
        shape.pop()
    count = int(np.prod(shape))
    dt = np.dtype(_NIFTI_DTYPES[datatype]).newbyteorder(endian)
    data = np.frombuffer(raw, dtype=dt, count=count, offset=int(vox_offset)).reshape(shape[::-1])    # x fastest
    data = data.astype(dt.newbyteorder("="))
    if scl_slope not in (0.0, 1.0) or scl_inter != 0.0:
        if scl_slope != 0.0 and not np.isnan(scl_slope):
            data = data.astype(np.float64) * scl_slope + scl_inter
    spacing = tuple(float(abs(p)) if p != 0 else 1.0 for p in pixdim[1:4])
    # RAS (NIfTI) -> LPS (ITK): negate the first two rows
    if sform_code > 0 and qform_code <= 0:
        rot = srow[:, :3] / np.maximum(np.linalg.norm(srow[:, :3], axis=0), 1e-20)
        off = srow[:, 3]
    elif qform_code > 0:
        rot = _quat_to_rot(*quatern)
        if pixdim[0] < 0:
            rot[:, 2] *= -1.0
        off = np.array(qoffset, np.float64)
    else:
        rot, off = np.eye(3), np.zeros(3)
    flip = np.diag([-1.0, -1.0, 1.0])
    direction = tuple(float(v) for v in (flip @ rot).reshape(-1))
    origin = tuple(float(v) for v in (flip @ off))
    return {"data": data, "spacing": spacing, "origin": origin, "direction": direction}


def write_nifti(data, filename, spacing=(1.0, 1.0, 1.0), origin=(0.0, 0.0, 0.0), direction=None):
    """[z,y,x] numpy array -> single-file NIfTI-1 with qform and sform set (spacing / origin / direction in ITK's LPS
    convention, as SimpleITK's SetSpacing / SetOrigin / SetDirection take them)."""
    arr = np.ascontiguousarray(data)
    if arr.dtype == np.bool_:
        arr = arr.astype(np.uint8)
    if arr.dtype not in _NIFTI_CODES:
        arr = arr.astype(np.float32 if arr.dtype.kind == "f" else np.int32)
    if arr.ndim != 3:
        raise ValueError("write_nifti expects a 3-D array [z,y,x]")
    flip = np.diag([-1.0, -1.0, 1.0])
    dmat = np.eye(3) if direction is None else np.asarray(direction, np.float64).reshape(3, 3)
    rot = flip @ dmat                                                   # LPS -> RAS
    off = flip @ np.asarray(origin, np.float64)
    qfac = 1.0
    r = rot.copy()
    if np.linalg.det(r) < 0:
        r[:, 2] *= -1.0
        qfac = -1.0
    b, c, d = _rot_to_quat(r)
    sp = [float(s) for s in spacing]
    hdr = bytearray(348)
    struct.pack_into("<i", hdr, 0, 348)
    struct.pack_into("<8h", hdr, 40, 3, arr.shape[2], arr.shape[1], arr.shape[0], 1, 1, 1, 1)
    struct.pack_into("<h", hdr, 70, _NIFTI_CODES[arr.dtype])
    struct.pack_into("<h", hdr, 72, arr.dtype.itemsize * 8)
    struct.pack_into("<8f", hdr, 76, qfac, sp[0], sp[1], sp[2], 0.0, 0.0, 0.0, 0.0)
    struct.pack_into("<f", hdr, 108, 352.0)
    struct.pack_into("<2f", hdr, 112, 1.0, 0.0)
    hdr[123] = 2                                                        # xyzt_units: millimetres
    struct.pack_into("<2h", hdr, 252, 1, 1)
    struct.pack_into("<3f", hdr, 256, b, c, d)
    struct.pack_into("<3f", hdr, 268, *[float(v) for v in off])
    srow = np.concatenate([rot * np.asarray(sp)[None, :], off[:, None]], 1)
    struct.pack_into("<12f", hdr, 280, *[float(v) for v in srow.reshape(-1)])
    hdr[344:348] = b"n+1\0"
    payload = bytes(hdr) + b"\0\0\0\0" + arr.astype(arr.dtype.newbyteorder("<")).tobytes()
    opener = gzip.open if str(filename).endswith(".gz") else open
    with opener(filename, "wb") as f:
        f.write(payload)


# -- PyMIC-shaped wrappers (io/image_read_write.py) -------------------------------------------------------------------
def load_nifty_volume_as_4d_array(filename):
    """image_read_write.py:9-37: {'data_array' [C,D,H,W], 'origin', 'spacing' (z,y,x), 'direction'}."""
    img = read_nifti(filename)
    data = img["data"]
    if data.ndim == 4:
        if data.shape[0] != 1:
            raise ValueError("unsupported image dim: 4 with %d frames" % data.shape[0])
    elif data.ndim == 3:
        data = data[None]
    else:
        raise ValueError("unsupported image dim: {0:}".format(data.ndim))
    sp = img["spacing"]
    return {"data_array": data, "origin": img["origin"], "spacing": (sp[2], sp[1], sp[0]), "direction": img["direction"]}


def load_image_as_nd_array(image_name):
    """image_read_write.py:69-90 for the formats the FPL+ recipe uses (.nii.gz / .nii / .npy)."""
    if image_name.endswith(".nii.gz") or image_name.endswith(".nii"):
        return load_nifty_volume_as_4d_array(image_name)
    if image_name.endswith(".npy"):
        return np.load(image_name, allow_pickle=True)
    raise ValueError("unsupported image format")


def load_volume(path):
    """One volume of a training-CSV row: a ``.npy`` array as stored, or the [D,H,W] data of a ``.nii`` / ``.nii.gz``
    file (``NpyVolumeDataset`` and ``datapath.load_train_csv``)."""
    if path.endswith(('.nii.gz', '.nii')):
        return load_nifty_volume_as_4d_array(path)['data_array'][0]
    return np.load(path)


def save_array_as_nifty_volume(data, image_name, reference_name=None):
    """image_read_write.py:92-108: [D,H,W] array, geometry copied from ``reference_name`` when given."""
    meta = {}
    if reference_name is not None:
        ref = read_nifti(reference_name)
        meta = {"spacing": ref["spacing"], "origin": ref["origin"], "direction": ref["direction"]}
    write_nifti(data, image_name, **meta)


def save_nd_array_as_image(data, image_name, reference_name=None):
    """image_read_write.py:130-148 for NIfTI outputs."""
    if image_name.endswith(".nii.gz") or image_name.endswith(".nii"):
        assert data.ndim == 3
        save_array_as_nifty_volume(data, image_name, reference_name)
    elif image_name.endswith(".npy"):
        np.save(image_name, data)
    else:
        raise ValueError("unsupported image format {0:}".format(image_name.split('.')[-1]))


# -- pixel weights (data/get_pixel_weight.py:12-28) -------------------------------------------------------------------
def pixel_weight_from_label_files(label_target, label_fake_source, out_name):
    """Two pseudo-label volumes of one target image (target-domain pass, fake-source pass) -> the agreement weight volume
    (1 where they agree, 0.5 where they differ), saved beside them with the target volume's geometry."""
    a = load_image_as_nd_array(label_target)["data_array"][0]
    b = load_image_as_nd_array(label_fake_source)["data_array"][0]
    w = 1.0 - 0.5 * (np.asarray(a) != np.asarray(b))
    save_nd_array_as_image(w, out_name, label_target if label_target.endswith((".nii", ".nii.gz")) else None)
    return w


# -- image weights + training CSV (README.md:74: the script is missing from the reference tree) ---------------------
def image_weight_table(sorted_uncertainty):
    """``fpl_uncertainty_sorted.npy`` rows ([value], name) (agent_seg.py:954-960) -> [(name, image_weight)] in the same
    (ascending-uncertainty) order: w = 1.01 - (u - u_min)/(u_max* - u_min), sentinel u == 1 -> 0.01 (SURVEY 8 a18;
    reproduces config_dual/data_vs/train_vs_t1s_wi+wp.csv from dataset/weight/cyc121_vst1s-gan.npy to 1e-16)."""
    from .fpl import image_weights
    rows = [(r[0], r[1]) for r in sorted_uncertainty]
    vals = [float(v[0]) if isinstance(v, (list, tuple, np.ndarray)) else float(v) for v, _n in rows]
    w = image_weights(vals)
    return [(str(n), float(wi)) for (_v, n), wi in zip(rows, w)]


def write_train_csv(path, rows, fields=("image", "label", "pixel_weight", "image_weight")):
    """The 4-column CSV NiftyDataset reads (io/nifty_dataset.py:60-75; config_dual/data_vs/train_vs_t1s_wi+wp.csv)."""
    with open(path, "w", newline="") as f:
        wr = csv.writer(f, delimiter=",", quotechar='"', quoting=csv.QUOTE_MINIMAL)
        wr.writerow(list(fields))
        for r in rows:
            wr.writerow(list(r))


def train_csv_from_uncertainty(sorted_npy, out_csv, label_of=None, pixel_weight_of=None):
    """The missing ``data/get image_weight.py``: sorted uncertainties -> image weights -> the final segmentor's training CSV.
    ``label_of`` / ``pixel_weight_of`` map an image path to its pseudo-label / pixel-weight path (default: same path, as
    in the shipped CSV)."""
    srt = np.load(sorted_npy, allow_pickle=True) if isinstance(sorted_npy, str) else sorted_npy
    table = image_weight_table(srt)
    label_of = label_of or (lambda n: n)
    pixel_weight_of = pixel_weight_of or (lambda n: n)
    rows = [(n, label_of(n), pixel_weight_of(n), repr(w)) for n, w in table]
    write_train_csv(out_csv, rows)
    return rows


# -- evaluation (util/evaluation_seg_train.py) ------------------------------------------------------------------------
def binary_dice(s, g):
    """evaluation_seg_train.py:21-50."""
    assert len(s.shape) == len(g.shape)
    s0 = np.multiply(s, g).sum()
    return (2.0 * s0 + 1e-5) / (s.sum() + g.sum() + 1e-5)


def get_edge_points(img):
    """evaluation_seg_train.py:83-99: the mask minus its 6-/4-connected erosion."""
    from scipy import ndimage
    strt = ndimage.generate_binary_structure(len(img.shape), 1)
    ero = ndimage.binary_erosion(img, strt)
    return np.asarray(img, np.uint8) - np.asarray(ero, np.uint8)


def binary_assd(s, g, spacing=None):
    """evaluation_seg_train.py:139-172: average symmetric surface distance, capped at 50.  The reference measures the
    distances with GeodisTK's 2-pass raster scan (lambda = 0, an approximation of the Euclidean distance transform); this
    uses scipy's exact Euclidean distance transform with the same spacing."""
    from scipy import ndimage
    s_edge, g_edge = get_edge_points(s), get_edge_points(g)
    dim = len(s.shape)
    assert dim == len(g.shape)
    spacing = [1.0] * dim if spacing is None else list(spacing)
    assert dim == len(spacing)
    ns, ng = s_edge.sum(), g_edge.sum()
    if ns == 0 or ng == 0:
        return 50
    s_dis = ndimage.distance_transform_edt(s_edge == 0, sampling=spacing)
    g_dis = ndimage.distance_transform_edt(g_edge == 0, sampling=spacing)
    assd = ((s_dis * g_edge).sum() + (g_dis * s_edge).sum()) / (ns + ng)
    return 50 if assd > 50 else assd


def evaluate_label_volumes(seg, gt, label_list, spacing=None, metrics=("dice", "assd")):
    """Per-class scores of one volume (the inner loop of evaluation_seg_train.py:evaluation): {metric: [score per label]}."""
    out = {}
    for m in metrics:
        fn = binary_dice if m == "dice" else (lambda a, b: binary_assd(a, b, spacing))
        out[m] = [float(fn(np.asarray(seg == lab, np.uint8), np.asarray(gt == lab, np.uint8))) for lab in label_list]
    return out


def evaluate_folder(pairs, label_list, out_csv=None, metric="dice"):
    """pairs: [(name, segmentation path, ground-truth path)] -> rows [name, class scores.., average]; mean / std rows and
    the CSV layout of evaluation_seg_train.py:560-575."""
    rows = []
    for name, s_name, g_name in pairs:
        s = load_image_as_nd_array(s_name)
        g = load_image_as_nd_array(g_name)
        sp = s.get("spacing") if isinstance(s, dict) else None
        s = s["data_array"][0] if isinstance(s, dict) else np.asarray(s)
        g = g["data_array"][0] if isinstance(g, dict) else np.asarray(g)
        sc = evaluate_label_volumes(s, g, label_list, sp, (metric,))[metric]
        rows.append([name] + sc + ([float(np.mean(sc))] if len(label_list) > 1 else []))
    scores = np.asarray([r[1:] for r in rows], np.float64)
    rows.append(["mean"] + list(scores.mean(0)))
    rows.append(["std"] + list(scores.std(0)))
    if out_csv:
        head = ["image"] + ["class_{0:}".format(i) for i in label_list] + (["average"] if len(label_list) > 1 else [])
        with open(out_csv, "w", newline="") as f:
            wr = csv.writer(f, delimiter=",", quotechar='"', quoting=csv.QUOTE_MINIMAL)
            wr.writerow(head)
            for r in rows:
                wr.writerow(r)
    return rows
