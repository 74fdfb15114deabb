"""Step-front data path: the on-disk latent format the reference trains from, and the loader that feeds `TrainStep`.

Reference: `ImageNetLatentDataset` (train_utils/datasets.py:240-304) reads an LMDB environment `<root>/<split>` with
keys `length` (decimal string), `z-{i}` (raw little-endian fp32 bytes of the VAE moments `[2C, R, R]`, written by
extract_latent.py:69-73,106) and `y-{i}` (decimal class index); `train.py:109-115` wraps it in a DataLoader
(`shuffle=False, drop_last=True`, batch = micro-batch x grad_accum) and `helper.get_one_hot` turns the class index
into the float one-hot the label embedder consumes.

The `lmdb` Python module is not part of this image, so `MdbReader` below is a read-only walker of LMDB's on-disk
B+tree (`data.mdb`: two meta pages, branch / leaf / overflow pages) written from the published file format; when
`lmdb` IS importable it is used instead.  PARITY UNPINNED against liblmdb itself (no liblmdb here to produce a
fixture): `tests/test_data.py` round-trips files produced by `write_mdb` / `MdbWriter` (the same format; `MdbWriter`
streams overflow values to disk, so a 1.28 M-image ImageNet extraction never holds its ~42 GB of moments in memory).

Nothing here runs on the GPU: batches are assembled in pinned host memory and copied by the caller; the arithmetic
that follows (moments -> latent, label dropout, noise injection) is `ops.step_front` (csrc/loss_optim.cu).
"""
from __future__ import annotations

import mmap
import os
import struct

import numpy as np
import torch

P_BRANCH, P_LEAF, P_OVERFLOW, P_META = 0x01, 0x02, 0x04, 0x08
F_BIGDATA = 0x01
MDB_MAGIC = 0xBEEFC0DE
PAGEHDR = 16
P_INVALID = (1 << 64) - 1


class MdbReader:
    """Read-only point lookups in an LMDB `data.mdb` (main database, default byte-wise key order, 64-bit build)."""

    def __init__(self, path):
        f = os.path.join(path, "data.mdb") if os.path.isdir(path) else path
        self._fh = open(f, "rb")
        self._mm = mmap.mmap(self._fh.fileno(), 0, access=mmap.ACCESS_READ)
        mm = self._mm
        magic, version = struct.unpack_from("<II", mm, PAGEHDR)
        if magic != MDB_MAGIC:
            raise IOError(f"{f}: not an LMDB data file (magic {magic:#x})")
        self.psize = struct.unpack_from("<I", mm, PAGEHDR + 24)[0]   # mm_dbs[FREE_DBI].md_pad holds the page size
        best = None
        for pg in (0, 1):                                            # the meta page with the newer transaction id wins
            base = pg * self.psize + PAGEHDR
            if struct.unpack_from("<I", mm, base)[0] != MDB_MAGIC:
                continue
            txnid = struct.unpack_from("<Q", mm, base + 128)[0]
            if best is None or txnid > best[0]:
                depth = struct.unpack_from("<H", mm, base + 78)[0]
                entries, root = struct.unpack_from("<QQ", mm, base + 104)
                best = (txnid, depth, entries, root)
        self.txnid, self.depth, self.entries, self.root = best

    def close(self):
        self._mm.close()
        self._fh.close()

    def _nodes(self, pgno):
        base = pgno * self.psize
        flags, lower = struct.unpack_from("<HH", self._mm, base + 10)
        n = (lower - PAGEHDR) // 2
        return base, flags, struct.unpack_from(f"<{n}H", self._mm, base + PAGEHDR)

    def _node(self, base, off):
        lo, hi, nflags, ksize = struct.unpack_from("<HHHH", self._mm, base + off)
        key = self._mm[base + off + 8: base + off + 8 + ksize]
        return lo, hi, nflags, key, base + off + 8 + ksize

    def get(self, key: bytes):
        if self.root == P_INVALID:
            return None
        pgno = self.root
        while True:
            base, flags, ptrs = self._nodes(pgno)
            if flags & P_BRANCH:
                lo_i, hi_i = 0, len(ptrs) - 1                       # node 0 of a branch page has an empty key (= -inf)
                while lo_i < hi_i:                                   # last node whose key <= the searched key
                    mid = (lo_i + hi_i + 1) // 2
                    if self._node(base, ptrs[mid])[3] <= key:
                        lo_i = mid
                    else:
                        hi_i = mid - 1
                lo, hi, nflags, _, _ = self._node(base, ptrs[lo_i])
                pgno = lo | (hi << 16) | (nflags << 32)
                continue
            if not flags & P_LEAF:
                raise IOError(f"page {pgno}: unexpected flags {flags:#x}")
            a, b = 0, len(ptrs) - 1
            while a <= b:
                mid = (a + b) // 2
                lo, hi, nflags, k, dpos = self._node(base, ptrs[mid])
                if k == key:
                    size = lo | (hi << 16)
                    if nflags & F_BIGDATA:
                        ov = struct.unpack_from("<Q", self._mm, dpos)[0]
                        start = ov * self.psize + PAGEHDR
                        return self._mm[start:start + size]
                    return self._mm[dpos:dpos + size]
                if k < key:
                    a = mid + 1
                else:
                    b = mid - 1
            return None


def _node(key, size, flags, payload):
    """Leaf node: (size lo, size hi, flags, key size), key, then the value (or the first overflow pgno, F_BIGDATA)."""
    return struct.pack("<HHHH", size & 0xFFFF, size >> 16, flags, len(key)) + key + payload


def _branch_node(key, pgno):
    return struct.pack("<HHHH", pgno & 0xFFFF, (pgno >> 16) & 0xFFFF, (pgno >> 32) & 0xFFFF, len(key)) + key


class MdbWriter:
    """Stream a fresh single-database LMDB file `<path>/data.mdb` (the layout extract_latent.py:60-106 writes with
    liblmdb).  `put(key, value)` appends values too large for a leaf node (every VAE moment) to the file at once as
    overflow pages; only `(key, pgno, length)` records and small inline values stay in memory.  `close()` builds the
    sorted leaf and branch pages after them and then writes the two meta pages at offsets 0 and psize.  Keys may come
    in any order; a key can be put once."""

    def __init__(self, path, psize=4096):
        os.makedirs(path, exist_ok=True)
        self.psize = psize
        self._f = open(os.path.join(path, "data.mdb"), "wb")
        self._f.write(bytes(2 * psize))          # meta pages 0 and 1, written by close()
        self._next = 2                           # next free page number
        self._nodes = {}                         # key -> leaf node bytes
        self._n_over = 0

    def _write_pages(self, buf):
        assert len(buf) % self.psize == 0
        pg = self._next
        self._f.write(buf)
        self._next += len(buf) // self.psize
        return pg

    def put(self, key, value):
        key, value = bytes(key), bytes(value)
        if key in self._nodes:
            raise KeyError(f"MdbWriter: key {key!r} was already put")
        psize = self.psize
        if 8 + len(key) + len(value) > psize // 2 - PAGEHDR:        # value goes to overflow pages
            npg = (PAGEHDR + len(value) + psize - 1) // psize
            buf = bytearray(npg * psize)
            struct.pack_into("<QHHI", buf, 0, self._next, 0, P_OVERFLOW, npg)
            buf[PAGEHDR:PAGEHDR + len(value)] = value
            ov = self._write_pages(buf)
            self._n_over += npg
            self._nodes[key] = _node(key, len(value), F_BIGDATA, struct.pack("<Q", ov))
        else:
            self._nodes[key] = _node(key, len(value), 0, value)

    def _page(self, flags, nodes):
        psize = self.psize
        buf = bytearray(psize)
        upper = psize
        ptrs = []
        for nd in nodes:
            upper -= len(nd) + (len(nd) & 1)
            buf[upper:upper + len(nd)] = nd
            ptrs.append(upper)
        lower = PAGEHDR + 2 * len(ptrs)
        assert lower <= upper
        struct.pack_into("<QHHHH", buf, 0, self._next, 0, flags, lower, upper)
        struct.pack_into(f"<{len(ptrs)}H", buf, PAGEHDR, *ptrs)
        return self._write_pages(buf)

    def _fits(self, nodes, used, nd):
        return PAGEHDR + 2 * (len(nodes) + 1) + used + len(nd) + (len(nd) & 1) <= self.psize

    def close(self):
        if self._f is None:
            return
        psize = self.psize
        keys = sorted(self._nodes)
        n_leaf = n_branch = 0
        level = []          # (first key, pgno)
        cur, used, first = [], 0, None
        for k in keys:
            nd = self._nodes.pop(k)
            if cur and not self._fits(cur, used, nd):
                level.append((first, self._page(P_LEAF, cur)))
                n_leaf += 1
                cur, used, first = [], 0, None
            if first is None:
                first = k
            cur.append(nd)
            used += len(nd) + (len(nd) & 1)
        if cur:
            level.append((first, self._page(P_LEAF, cur)))
            n_leaf += 1
        depth = 1 if level else 0
        while len(level) > 1:
            nxt, cur, used, first = [], [], 0, None
            for k, pg in level:
                nd = _branch_node(b"" if not cur else k, pg)     # node 0 of a branch page has an empty key
                if cur and not self._fits(cur, used, nd):
                    nxt.append((first, self._page(P_BRANCH, cur)))
                    n_branch += 1
                    cur, used, first = [], 0, None
                    nd = _branch_node(b"", pg)
                if first is None:
                    first = k
                cur.append(nd)
                used += len(nd) + (len(nd) & 1)
            nxt.append((first, self._page(P_BRANCH, cur)))
            n_branch += 1
            level = nxt
            depth += 1
        root = level[0][1] if level else P_INVALID
        last_pg = self._next - 1
        for m in (0, 1):
            buf = bytearray(psize)
            struct.pack_into("<QHHI", buf, 0, m, 0, P_META, 0)
            b = PAGEHDR
            struct.pack_into("<IIQQ", buf, b, MDB_MAGIC, 1, 0, max(1 << 20, (last_pg + 1) * psize))
            struct.pack_into("<IHHQQQQQ", buf, b + 24, psize, 0, 0, 0, 0, 0, 0, P_INVALID)        # free DB (empty)
            struct.pack_into("<IHHQQQQQ", buf, b + 72, 0, 0, depth, n_branch, n_leaf, self._n_over, len(keys), root)
            struct.pack_into("<QQ", buf, b + 120, last_pg, 1 if m == 1 else 0)
            self._f.seek(m * psize)
            self._f.write(buf)
        self._f.close()
        self._f = None

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()


def write_mdb(path, items, psize=4096):
    """Bulk-load `items` (dict bytes -> bytes) into a fresh single-database LMDB file `<path>/data.mdb` (tests and
    synthetic datasets) through `MdbWriter`."""
    with MdbWriter(path, psize) as w:
        for k in sorted(items):
            w.put(k, items[k])


def center_crop_arr(pil_image, image_size):
    """The reference's image preprocessing (train_utils/datasets.py:19-37, ADM's center crop): halve with BOX filtering
    while the short side is at least twice `image_size`, resize with BICUBIC so the short side is `image_size`, then crop
    the centre square.  Returns a PIL image of `image_size` x `image_size`."""
    from PIL import Image
    img = pil_image
    while min(img.size) >= 2 * image_size:
        img = img.resize((img.width // 2, img.height // 2), resample=Image.BOX)
    s = image_size / min(img.size)
    img = img.resize((round(img.width * s), round(img.height * s)), resample=Image.BICUBIC)
    top, left = (img.height - image_size) // 2, (img.width - image_size) // 2
    return Image.fromarray(np.asarray(img)[top:top + image_size, left:left + image_size])


def write_latent_lmdb(root, moments, labels, split="train"):
    """`<root>/<split>` in the layout extract_latent.py produces: z-{i} raw fp32 moments, y-{i} class index, length."""
    items = {b"length": str(len(labels)).encode()}
    for i, (z, y) in enumerate(zip(moments, labels)):
        items[f"z-{i}".encode()] = np.ascontiguousarray(z, dtype="<f4").tobytes()
        items[f"y-{i}".encode()] = str(int(y)).encode()
    write_mdb(os.path.join(root, split), items)


class ImageNetLatentDataset:
    """train_utils/datasets.py:240-304 (latent + class index; the `feat_path` / `xflip` variants are not used by any
    shipped config and raise).  `__getitem__` -> (moments float32 [2C, R, R], one-hot float32 [num_classes])."""

    def __init__(self, path, resolution=32, num_channels=4, split="train", num_classes=1000, feat_path=None,
                 feat_dim=0, xflip=False):
        if feat_path is not None or feat_dim or xflip:
            raise NotImplementedError("feature-conditioned / x-flipped latent datasets are outside the MaskDiT hot path")
        self._path = os.path.join(path, split)
        if not os.path.exists(os.path.join(self._path, "data.mdb")):
            raise FileNotFoundError(f"no LMDB latent dataset at {self._path} (expected data.mdb; "
                                    "reference layout: extract_latent.py)")
        self.resolution, self.num_channels, self.num_classes = resolution, num_channels, num_classes
        try:
            import lmdb  # noqa: F401 - liblmdb when the module exists
            self._env = lmdb.open(self._path, readonly=True, lock=False, create=False)
            self._txn = self._env.begin(write=False)
            self._get = self._txn.get
        except ImportError:
            self._rd = MdbReader(self._path)
            self._get = self._rd.get
        self.length = int(bytes(self._get(b"length")).decode())

    def __len__(self):
        return self.length

    def raw(self, idx):
        z = np.frombuffer(bytes(self._get(f"z-{idx}".encode())), dtype="<f4").reshape(
            -1, self.resolution, self.resolution).copy()                      # datasets.py:289: .copy()
        return z, int(bytes(self._get(f"y-{idx}".encode())).decode())

    def __getitem__(self, idx):
        z, y = self.raw(idx)
        onehot = np.zeros(self.num_classes, dtype=np.float32)   # helper.get_one_hot (train_utils/helper.py:30-33)
        onehot[y] = 1
        return z, onehot


def batches(dataset, batch, rank=0, world=1, start=0, pin=True):
    """Sequential, rank-strided, drop-last batches forever (train.py:109-115: `shuffle=False, drop_last=True`; the
    reference shards by accelerate's loader wrapper).  Yields pinned host tensors (moments [B,2C,R,R], labels [B,nc])."""
    n = len(dataset)
    per_epoch = n // (batch * world)
    if per_epoch == 0:
        raise ValueError(f"dataset of {n} items is smaller than one global batch ({batch} x {world})")
    z0, y0 = dataset[0]
    zb = torch.empty((batch, *z0.shape), dtype=torch.float32)
    yb = torch.empty((batch, y0.shape[0]), dtype=torch.float32)
    if pin and torch.cuda.is_available():
        zb, yb = zb.pin_memory(), yb.pin_memory()
    it = start
    while True:
        b = it % per_epoch
        base = (b * world + rank) * batch
        for j in range(batch):
            z, y = dataset[base + j]
            zb[j] = torch.from_numpy(np.ascontiguousarray(z))
            yb[j] = torch.from_numpy(y)
        yield zb, yb
        it += 1


# ---- WebDataset shards (lmdb2wds.py:26, train_wds.py:58-64) ------------------------------------------------------------
def write_wds_shard(path, moments, labels, start=0):
    """One tar shard in the layout lmdb2wds.py writes: `<key>.latent` = pickle of the [2C,R,R] float32 array,
    `<key>.cls` = the class index as ASCII (webdataset's default encoding of an int)."""
    import io
    import pickle
    import tarfile
    with tarfile.open(path, "w") as tf:
        for i, (z, y) in enumerate(zip(moments, labels)):
            key = f"{start + i:07d}"
            for ext, payload in (("latent", pickle.dumps(np.ascontiguousarray(z, dtype=np.float32))),
                                 ("cls", str(int(y)).encode())):
                ti = tarfile.TarInfo(f"{key}.{ext}")
                ti.size = len(payload)
                tf.addfile(ti, io.BytesIO(payload))


def wds_samples(shards, rank=0, world=1, num_classes=1000):
    """Iterate (moments float32 [2C,R,R], one-hot float32 [num_classes]) over this rank's shards, forever
    (train_wds.py:44-48 splits the shard list `data_list[rank::world]`; :58-64 decodes `latent` with pickle and `cls`
    as a decimal string).  Pickle is executed: shards must be trusted, as in the reference."""
    import pickle
    import tarfile
    mine = list(shards)[rank::world]
    if not mine:
        raise ValueError(f"{len(list(shards))} shards cannot be split over {world} ranks")
    while True:
        for path in mine:
            with tarfile.open(path, "r") as tf:
                cur, item = None, {}
                for m in tf:
                    if not m.isfile():
                        continue
                    key, _, ext = m.name.rpartition(".")
                    if key != cur and item:
                        item = {}
                    cur = key
                    item[ext] = tf.extractfile(m).read()
                    if "latent" in item and "cls" in item:
                        z = np.asarray(pickle.loads(item["latent"]), dtype=np.float32)
                        onehot = np.zeros(num_classes, dtype=np.float32)
                        onehot[int(item["cls"].decode("utf-8"))] = 1
                        item = {}
                        yield z, onehot


def wds_batches(shards, batch, rank=0, world=1, num_classes=1000, pin=True):
    """Drop-last batches of pinned host tensors from WebDataset shards (the loader train_wds.py:66-95 builds)."""
    it = wds_samples(shards, rank, world, num_classes)
    z0, y0 = next(it)
    zb = torch.empty((batch, *z0.shape), dtype=torch.float32)
    yb = torch.empty((batch, y0.shape[0]), dtype=torch.float32)
    if pin and torch.cuda.is_available():
        zb, yb = zb.pin_memory(), yb.pin_memory()
    pending = [(z0, y0)]
    while True:
        for j in range(batch):
            z, y = pending.pop() if pending else next(it)
            zb[j] = torch.from_numpy(z)
            yb[j] = torch.from_numpy(y)
        yield zb, yb
