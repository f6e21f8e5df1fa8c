"""Host-side value objects accepted by the drop-in managers (reference: shapes.py).

The managers only read ``.width .height .gt_boxes[*].corners/.obj_cls/.resize()
.cache_key .data`` (reference: shapes.py:5-132,187-305), so any duck-typed
object works, including the reference's own ``shapes.Image``.  ``Image`` can be
built from in-memory pixels or from an ``image_path`` (lazy ``cv2.imread`` like
the reference); ``.data`` is the reference's host path (cv2 resize + flip),
``.data_device()`` / ``.preprocessed_device()`` do the resize, flip and mean
subtraction on the GPU (SURVEY 8f-4, `ops.image_resize_cubic`); `preprocessed_batch_device` does it for a batch of
differently sized images in one padded device call (`ops.image_resize_cubic_ragged`).
"""
import numpy as np


class Box:
    """Axis-aligned box, corners [x1, y1, x2, y2] (reference: shapes.py:307-408)."""
    __slots__ = ("x1", "y1", "x2", "y2")

    def __init__(self, x1, y1, x2, y2):
        self.x1, self.y1, self.x2, self.y2 = x1, y1, x2, y2

    @staticmethod
    def from_center_dims_int(x_center, y_center, width, height):
        """integer anchor box around a centre: x1 = cx - w // 2, x2 = x1 + w (reference: shapes.py:309-323)."""
        left, top = x_center - width // 2, y_center - height // 2
        return Box(left, top, left + width, top + height)

    @staticmethod
    def from_corners(coords):
        return Box(*coords)

    @property
    def width(self):
        return self.x2 - self.x1

    @property
    def height(self):
        return self.y2 - self.y1

    @property
    def x_center(self):
        return (self.x2 + self.x1) / 2

    @property
    def y_center(self):
        return (self.y1 + self.y2) / 2

    @property
    def corners(self):
        return np.array([self.x1, self.y1, self.x2, self.y2])

    @property
    def corner_dims(self):
        return np.array([self.x1, self.y1, self.width, self.height])

    @property
    def center_dims(self):
        return np.array([self.x_center, self.y_center, self.width, self.height])

    def resize(self, ratio):
        return Box(self.x1 * ratio, self.y1 * ratio, self.x2 * ratio, self.y2 * ratio)

    def horizontal_flip(self, image_width):
        """the same box in the horizontally mirrored image (reference: shapes.py:292-300)."""
        return Box(image_width - self.x2, self.y1, image_width - self.x1, self.y2)

    def __repr__(self):
        return "Box(%r, %r, %r, %r)" % (self.x1, self.y1, self.x2, self.y2)


class GroundTruthBox:
    """Labelled object (reference: shapes.py:187-305)."""
    __slots__ = ("obj_cls", "difficult", "box")

    def __init__(self, obj_cls, difficult, box):
        self.obj_cls, self.difficult, self.box = obj_cls, difficult, box

    x1 = property(lambda self: self.box.x1)
    y1 = property(lambda self: self.box.y1)
    x2 = property(lambda self: self.box.x2)
    y2 = property(lambda self: self.box.y2)
    width = property(lambda self: self.box.width)
    height = property(lambda self: self.box.height)
    x_center = property(lambda self: self.box.x_center)
    y_center = property(lambda self: self.box.y_center)
    corner_dims = property(lambda self: self.box.corner_dims)
    center_dims = property(lambda self: self.box.center_dims)

    @property
    def corners(self):
        return self.box.corners

    def resize(self, ratio):
        return GroundTruthBox(self.obj_cls, self.difficult, self.box.resize(ratio))

    def horizontal_flip(self, image_width):
        return GroundTruthBox(self.obj_cls, self.difficult, self.box.horizontal_flip(image_width))


class Image:
    """Image metadata + pixels (reference: shapes.py:5-132).  Pixels come from `data` (an in-memory BGR uint8 array of
    ANY size: it is resized to width x height on access, like the reference resizes what it reads from disk) or, lazily,
    from `image_path`."""

    def __init__(self, name, width, height, gt_boxes=(), flipped=False, data=None, image_path=None):
        self.name, self.width, self.height = name, width, height
        self.gt_boxes, self.flipped, self._data, self.image_path = list(gt_boxes), flipped, data, image_path

    @property
    def cache_key(self):
        return self.name + str(self.flipped)

    def _raw(self):
        if self._data is not None:
            return self._data
        if self.image_path is None:
            raise ValueError("image %s carries no pixels" % self.name)
        import cv2
        img = cv2.imread(self.image_path)
        if img is None:
            raise IOError("cannot read %s" % self.image_path)
        return img

    @property
    def data(self):
        """shapes.py:19-29 on the host: the pixels resized (INTER_CUBIC) to width x height and mirrored when flipped.
        In-memory pixels that already have that size are returned as they are (they were resized by the caller)."""
        img = self._raw()
        if self.image_path is None and (img.ndim < 2 or img.shape[:2] == (self.height, self.width) or img.dtype != np.uint8):
            return img                                  # synthetic / already prepared arrays (tests, bench)
        import cv2
        img = cv2.resize(img, (self.width, self.height), interpolation=cv2.INTER_CUBIC)
        return cv2.flip(img, 1) if self.flipped and self.image_path is not None else img

    def data_device(self, mean=None, want_u8=True):
        """The same pixels computed on the GPU from the raw decoded image (one H2D of the uint8 pixels): returns the
        (height,width,C) u8 CUDA tensor, or with `mean` the float32 mean-subtracted tensor as well (ops.image_resize_cubic).
        Within one grey level of `.data` (OpenCV's own SIMD / generic code paths differ by as much, oracle/image_oracle.py).
        A path-backed JPEG file the device decoder supports is decoded on the device (ops.jpeg_decode, bit-exact with
        cv2.imread), and its compressed bytes are what is uploaded."""
        from . import ops
        from .runtime import get_context
        files = _jpeg_files([self])
        if files is not None:
            packed, _, _, status = ops.jpeg_decode([files[0][0]])
            h, w = files[0][1]
            dev = packed[:h * w * 3].view(1, h, w, 3)
        else:
            raw = np.ascontiguousarray(self._raw())
            if raw.dtype != np.uint8 or raw.ndim != 3:
                raise TypeError("data_device needs (H,W,C) uint8 pixels")
            dev = get_context().to_device(raw[None])
        out = ops.image_resize_cubic(dev, self.height, self.width, flip=self.flipped and self.image_path is not None,
                                     mean=mean, want_u8=want_u8)
        if files is not None and int(status[0]) != 0:
            return _host_decoded(self).data_device(mean=mean, want_u8=want_u8)   # corrupt data: cv2's own recovery
        return tuple(t[0] for t in out) if isinstance(out, tuple) else out[0]

    def preprocessed_device(self, mean=None):
        """float32 (1,height,width,C) CUDA tensor = resized (+ mirrored) BGR pixels minus the ImageNet means: what
        `batched_image` feeds the backbone (det_util.py:36, resnet.py:64-75), without leaving the device."""
        from . import ops
        return self.data_device(mean=ops.IMAGENET_MEAN_BGR if mean is None else mean, want_u8=False)[None]

    def resize(self, ratio):
        w, h = int(round(ratio * self.width)), int(round(ratio * self.height))
        return Image(self.name, w, h, [g.resize(ratio) for g in self.gt_boxes], self.flipped, self._data, self.image_path)

    def resize_within_bounds(self, min_size, max_size):
        short, long_ = min(self.width, self.height), max(self.width, self.height)
        r_min = min_size / short
        ratio = max_size / long_ if r_min * long_ > max_size else r_min
        return self.resize(ratio), ratio

    def horizontal_flip(self):
        """mirrored copy: boxes flipped about the image width, `flipped` toggled, so `cache_key` differs
        (reference: shapes.py:126-132,227-234).  In-memory pixels are mirrored here; pixels read from `image_path` are
        mirrored on access, like the reference does."""
        flipped = None if self._data is None or self.image_path is not None else self._data[:, ::-1]
        if self.image_path is not None:
            flipped = self._data
        return Image(self.name, self.width, self.height, [g.horizontal_flip(self.width) for g in self.gt_boxes],
                     not self.flipped, flipped, self.image_path)

    @property
    def num_gt_boxes(self):
        return len(self.gt_boxes)


def _jpeg_files(images):
    """[(file bytes, (h, w))] when every image is path-backed (no in-memory pixels) and every file is a JPEG the device
    decoder supports, else None."""
    from . import ops
    if any(img._data is not None or img.image_path is None for img in images):
        return None
    out = []
    for img in images:
        try:
            with open(img.image_path, "rb") as f:
                data = f.read()
        except OSError:
            return None
        hw = ops.jpeg_supported(data)
        if hw is None:
            return None
        out.append((data, hw))
    return out


def _host_decoded(img):
    """`img` with its pixels read by cv2.imread (mirrored on access like a path-backed image)."""
    return Image(img.name, img.width, img.height, img.gt_boxes, img.flipped, img._raw(), img.image_path)


def preprocessed_batch_device(images, mean=None, pad_to=None):
    """`Image.preprocessed_device` for a batch of differently sized images in one device call: every image is resized
    (and mirrored, under the rule of `data_device`) to its own height x width, minus the means, into one padded float32
    (B,H,W,C) CUDA tensor whose padding is zero.  (H, W) = the largest image, or `pad_to` (which must hold every image).
    Returns (padded, extents (B,2) i32 (height, width) on the device).  When every image is a path-backed JPEG file
    the device decoder supports, the compressed files are uploaded with one copy and decoded on the device
    (`ops.jpeg_decode`, bit-exact with cv2.imread); otherwise the raw pixels are read with cv2.imread, packed on the host
    and uploaded with one copy (`ops.pack_images`).  The target sizes and mirror flags take one more upload;
    `ops.image_resize_cubic_ragged` does the rest."""
    from . import ops
    images = list(images)
    if not images:
        raise ValueError("preprocessed_batch_device needs at least one image")
    sizes = np.array([(img.height, img.width) for img in images], np.int32).reshape(-1, 2)
    height, width = (int(v) for v in sizes.max(axis=0))
    if pad_to is not None:
        ph, pw = (int(v) for v in pad_to)
        if ph < height or pw < width:
            raise ValueError("pad_to %s is smaller than the largest image (%d, %d)" % ((ph, pw), height, width))
        height, width = ph, pw
    import torch
    from .runtime import get_context
    files = _jpeg_files(images)
    status = None
    if files is not None:
        src, offsets, src_sizes, status = ops.jpeg_decode([f for f, _ in files])
        channels = 3
    else:
        raws = [img._raw() for img in images]
        src, offsets, src_sizes = ops.pack_images(raws)
        channels = raws[0].shape[2]
    # target size and mirror flag of every image in one upload; the source sizes come with the sources
    flip = np.array([[img.flipped and img.image_path is not None] for img in images], np.int32)
    meta = get_context(src.device).to_device(np.concatenate([sizes, flip], axis=1))
    extents = meta[:, :2].contiguous()
    geom = torch.cat([src_sizes, extents], dim=1)
    mean = ops.IMAGENET_MEAN_BGR if mean is None else mean
    out = ops.image_resize_cubic_ragged(src, offsets, geom, height, width, flip=meta[:, 2].to(torch.uint8), mean=mean,
                                        want_u8=False, channels=channels)
    if status is not None and bool((status != 0).any()):
        # corrupt entropy data in some file: cv2.imread's own recovery defines those pixels
        return preprocessed_batch_device([_host_decoded(img) for img in images], mean=mean, pad_to=pad_to)
    return out, extents
