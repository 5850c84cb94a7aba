"""Minimal pure-Python reader for netCDF-4 (HDF5) files -- enough for CDO weight files and CF fields.

The reference opens weight files with ``xarray.open_dataset(..., engine="netcdf4")``
(/root/reference/smmregrid/cdogenerate.py:296) and CDO writes them as netCDF-4 when asked to
(``-f nc4``, cdogenerate.py:381) or when they are too large for the classic format.  Neither
``netCDF4`` nor ``h5py`` is a dependency of this package, so the subset of the HDF5 file format
that the netCDF-4 library produces is read here directly:

* superblock versions 0-3; object headers version 1 and 2 (with continuation blocks);
* groups as symbol tables (B-tree v1 + local heap) or link messages, compact or dense (fractal heap
  + B-tree v2);
* attributes in the header or dense (fractal heap + B-tree v2), fixed- and variable-length strings,
  integers, floats, object references (``DIMENSION_LIST`` through the global heap);
* data layouts version 3 (compact, contiguous, chunked through a B-tree v1) and version 4 with a
  single chunk or an implicit index; filters deflate, shuffle and fletcher32;
* the netCDF-4 conventions on top: dimension scales, ``_Netcdf4Dimid``, ``_Netcdf4Coordinates``,
  ``_nc4_non_coord_`` names, phony dimensions for files without scales.

User-defined types, compound data, external storage and the HDF5 1.10 chunk indexes that the
netCDF library never selects raise ``NotImplementedError`` naming the feature.  Only the root group
is exposed as netCDF variables (``File.groups`` lists the names of the others).

    with nc4.File(path) as f:
        f.dimensions            # {"num_links": 7128000, ...} in dimension-id order
        f.attrs                 # global attributes
        v = f.variables["remap_matrix"]; v.dims, v.shape, v.dtype, v.attrs
        a = v[...]              # numpy array (whole variable; v[idx] indexes the loaded array)
"""
from __future__ import annotations

import mmap
import struct
import zlib

import numpy as np

MAGIC = b"\x89HDF\r\n\x1a\n"

_UNDEF = {4: 0xFFFFFFFF, 8: 0xFFFFFFFFFFFFFFFF, 2: 0xFFFF}


def is_hdf5(path) -> bool:
    with open(path, "rb") as fh:
        return fh.read(8) == MAGIC


def _log2(n: int) -> int:
    return int(n).bit_length() - 1


def _enc_size(limit: int) -> int:
    """bytes the library uses to store values up to `limit` (H5VM_limit_enc_size)"""
    return _log2(max(int(limit), 1)) // 8 + 1


class _Datatype:
    """Parsed datatype message (only what is needed to decode values)."""

    def __init__(self, buf: bytes):
        self.cls = buf[0] & 0x0F
        self.version = buf[0] >> 4
        bits = buf[1:4]
        self.size = struct.unpack_from("<I", buf, 4)[0]
        self.base = None
        self.dtype = None
        self.is_vlen_string = False
        if self.cls == 0:                           # fixed point
            order = ">" if bits[0] & 1 else "<"
            kind = "i" if bits[0] & 8 else "u"
            self.dtype = np.dtype(f"{order}{kind}{self.size}")
        elif self.cls == 1:                         # floating point
            order = ">" if bits[0] & 1 else "<"
            self.dtype = np.dtype(f"{order}f{self.size}")
        elif self.cls == 3:                         # fixed-length string
            self.dtype = np.dtype(f"S{self.size}")
        elif self.cls == 7:                         # reference
            self.dtype = np.dtype(f"<u{self.size}")
        elif self.cls == 9:                         # variable length
            self.is_vlen_string = (bits[0] & 0x0F) == 1
            self.base = _Datatype(buf[8:])
        elif self.cls == 8:                         # enum: values of the base type
            self.base = _Datatype(buf[8:])
            self.dtype = self.base.dtype
        elif self.cls == 10:                        # array
            raise NotImplementedError("HDF5 array datatypes")
        elif self.cls == 6:
            raise NotImplementedError("HDF5 compound datatypes")
        else:
            raise NotImplementedError(f"HDF5 datatype class {self.cls}")


class Variable:
    """One netCDF variable: metadata now, data on first access."""

    def __init__(self, f: "File", name: str, obj: dict):
        self._f = f
        self._obj = obj
        self.name = name
        self.shape = tuple(obj["shape"])
        self.dtype = obj["dtype"].dtype.newbyteorder("=") if obj["dtype"].dtype is not None else None
        self.attrs = {k: v for k, v in obj["attrs"].items() if k not in _HIDDEN_ATTRS}
        self.dims: tuple = ()
        self._data = None

    @property
    def ndim(self):
        return len(self.shape)

    @property
    def size(self):
        return int(np.prod(self.shape, dtype=np.int64)) if self.shape else 1

    def read(self) -> np.ndarray:
        if self._data is None:
            if self._f._b is None:
                raise ValueError(f"{self._f.path} is closed")
            try:
                self._data = self._f._read_dataset(self._obj)
            except (struct.error, IndexError, ValueError, TypeError, OverflowError, MemoryError, zlib.error) as e:
                raise OSError(f"{self._f.path}: variable {self.name}: damaged HDF5 file "
                              f"({type(e).__name__}: {e})") from e
        return self._data

    def __getitem__(self, idx):
        return self.read()[idx]

    def decoded(self) -> np.ndarray:
        """Values as ``xarray.open_dataset`` hands them to the reference (mask_and_scale):
        ``_FillValue`` / ``missing_value`` -> NaN, then ``scale_factor`` / ``add_offset``."""
        a = self.read()
        fills = [self.attrs[k] for k in ("_FillValue", "missing_value") if k in self.attrs]
        scale, offset = self.attrs.get("scale_factor"), self.attrs.get("add_offset")
        if not fills and scale is None and offset is None:
            return a
        out = a.astype(np.float32 if a.dtype.kind == "f" and a.dtype.itemsize <= 4 and scale is None and
                       offset is None else np.float64)
        for fv in fills:
            fv = np.asarray(fv).reshape(-1)[0]
            out[a == fv] = np.nan
        if scale is not None:
            out *= np.float64(scale)
        if offset is not None:
            out += np.float64(offset)
        return out

    def packing(self):
        """``CFPacking`` of this variable (None when it is not packed), so that its raw values are
        decoded inside the kernels: ``rg.regrid(var.read(), packing=var.packing())``."""
        from .packing import CFPacking
        return CFPacking.from_attrs(self.attrs, self.dtype)

    def __array__(self, dtype=None, copy=None):
        a = self.read()
        return a.astype(dtype) if dtype is not None else a

    def __repr__(self):
        return f"<nc4.Variable {self.name}{self.dims} {self.dtype} {self.shape}>"


_HIDDEN_ATTRS = {"DIMENSION_LIST", "REFERENCE_LIST", "CLASS", "NAME", "_Netcdf4Dimid", "_Netcdf4Coordinates",
                 "_nc3_strict", "_NCProperties"}
_NOT_A_VAR = "This is a netCDF dimension but not a netCDF variable."


class File:
    def __init__(self, path):
        self.path = str(path)
        self._fh = open(self.path, "rb")
        try:
            self._b = mmap.mmap(self._fh.fileno(), 0, access=mmap.ACCESS_READ)
        except ValueError:
            self._fh.close()
            raise OSError(f"{self.path}: empty file")
        try:
            self._open()
        except NotImplementedError:
            self.close()
            raise
        except (struct.error, IndexError, ValueError, TypeError, OverflowError, MemoryError, zlib.error, RecursionError) as e:
            self.close()                            # truncated or damaged: report it as such
            raise OSError(f"{self.path}: damaged HDF5 file ({type(e).__name__}: {e})") from e
        except Exception:
            self.close()
            raise

    # ------------------------------------------------------------------ plumbing
    def close(self):
        if getattr(self, "_b", None) is not None:
            self._b.close()
            self._b = None
        if getattr(self, "_fh", None) is not None:
            self._fh.close()
            self._fh = None

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def _u(self, off: int, n: int) -> int:
        return int.from_bytes(self._b[off:off + n], "little")

    def _addr(self, off: int) -> int:
        return self._u(off, self._O) + self._base

    def _is_undef(self, off: int, n: int | None = None) -> bool:
        n = n or self._O
        return self._b[off:off + n] == b"\xff" * n

    def _fail(self, what: str):
        raise OSError(f"{self.path}: not a readable HDF5 file ({what})")

    # ------------------------------------------------------------------ superblock
    def _open(self):
        b = self._b
        sb = 0
        while b[sb:sb + 8] != MAGIC:               # the superblock may sit at 512, 1024, ...
            sb = 512 if sb == 0 else sb * 2
            if sb + 8 > len(b):
                self._fail("no superblock")
        ver = b[sb + 8]
        self._base = 0
        if ver in (0, 1):
            self._O, self._L = b[sb + 13], b[sb + 14]
            p = sb + 24 + (4 if ver == 1 else 0)
            self._base = self._u(p, self._O)
            p += 4 * self._O
            root = self._u(p + self._O, self._O) + self._base     # symbol table entry: name offset, header address
        elif ver in (2, 3):
            self._O, self._L = b[sb + 9], b[sb + 10]
            p = sb + 12
            self._base = self._u(p, self._O)
            root = self._u(p + 3 * self._O, self._O) + self._base
        else:
            self._fail(f"superblock version {ver}")
        self._gcol: dict = {}
        self._objs: dict = {}
        rootobj = self._object(root)
        self.attrs = {k: v for k, v in rootobj["attrs"].items() if k not in _HIDDEN_ATTRS}
        self._netcdf_view(rootobj)

    # ------------------------------------------------------------------ object headers
    def _messages(self, addr: int):
        """(type, flags, bytes) of every message of the object header at `addr`."""
        b = self._b
        out = []
        if b[addr:addr + 4] == b"OHDR":
            if b[addr + 4] != 2:
                self._fail("object header version")
            fl = b[addr + 5]
            p = addr + 6
            if fl & 0x20:
                p += 16
            if fl & 0x10:
                p += 4
            n = 1 << (fl & 3)
            size0 = self._u(p, n)
            p += n
            blocks = [(p, p + size0)]
            hdr = 4 + (2 if fl & 0x04 else 0)
            while blocks:
                p, end = blocks.pop(0)
                while p + hdr <= end:
                    mtype = b[p]
                    msize = self._u(p + 1, 2)
                    mflags = b[p + 3]
                    d = p + hdr
                    if d + msize > end:
                        break
                    body = bytes(b[d:d + msize])
                    if mtype == 0x10:
                        co, cl = self._u(d, self._O) + self._base, self._u(d + self._O, self._L)
                        if b[co:co + 4] != b"OCHK":
                            self._fail("object header continuation")
                        blocks.append((co + 4, co + cl - 4))
                    elif mtype != 0:
                        out.append((mtype, mflags, body))
                    p = d + msize
        else:
            if b[addr] != 1:
                self._fail(f"object header at {addr}")
            nmsg = self._u(addr + 2, 2)
            size0 = self._u(addr + 8, 4)
            blocks = [(addr + 16, addr + 16 + size0)]
            while blocks and nmsg > 0:
                p, end = blocks.pop(0)
                while p + 8 <= end and nmsg > 0:
                    mtype = self._u(p, 2)
                    msize = self._u(p + 2, 2)
                    mflags = b[p + 4]
                    d = p + 8
                    body = bytes(b[d:d + msize])
                    nmsg -= 1
                    if mtype == 0x10:
                        co, cl = self._u(d, self._O) + self._base, self._u(d + self._O, self._L)
                        blocks.append((co, co + cl))
                    elif mtype != 0:
                        out.append((mtype, mflags, body))
                    p = d + msize
        return out

    def _object(self, addr: int) -> dict:
        if addr in self._objs:
            return self._objs[addr]
        obj = {"addr": addr, "attrs": {}, "links": {}, "shape": None, "dtype": None, "layout": None,
               "filters": [], "fill": None, "is_group": False, "maxshape": None}
        self._objs[addr] = obj
        for mtype, mflags, m in self._messages(addr):
            if mflags & 0x02:                       # shared message: only user-defined types use these
                continue
            if mtype == 0x01:
                obj["shape"], obj["maxshape"] = self._dataspace(m)
            elif mtype == 0x03:
                try:
                    obj["dtype"] = _Datatype(m)
                except NotImplementedError as e:
                    obj["dtype_error"] = str(e)
            elif mtype == 0x05:
                obj["fill"] = self._fillvalue(m)
            elif mtype == 0x08:
                obj["layout"] = m
            elif mtype == 0x0B:
                obj["filters"] = self._filters(m)
            elif mtype == 0x0C:
                self._attribute(m, obj["attrs"])
            elif mtype == 0x06:
                obj["is_group"] = True
                self._link(m, obj["links"])
            elif mtype == 0x02:                     # link info: dense links
                obj["is_group"] = True
                p = 2 + (8 if m[1] & 1 else 0)
                if not self._undef_bytes(m[p:p + self._O]):
                    heap = int.from_bytes(m[p:p + self._O], "little") + self._base
                    bt = int.from_bytes(m[p + self._O:p + 2 * self._O], "little") + self._base
                    for rec in self._btree2(bt):
                        body = self._heap_object(heap, rec[4:])        # type 5 record: hash, heap id
                        self._link(body, obj["links"])
            elif mtype == 0x11:                     # symbol table (old-style group)
                obj["is_group"] = True
                bt = int.from_bytes(m[:self._O], "little") + self._base
                hp = int.from_bytes(m[self._O:2 * self._O], "little") + self._base
                self._symbol_table(bt, hp, obj["links"])
            elif mtype == 0x15:                     # attribute info: dense attributes
                p = 2 + (2 if m[1] & 1 else 0)
                if not self._undef_bytes(m[p:p + self._O]):
                    heap = int.from_bytes(m[p:p + self._O], "little") + self._base
                    bt = int.from_bytes(m[p + self._O:p + 2 * self._O], "little") + self._base
                    for rec in self._btree2(bt):
                        if rec[self._heap(heap)["id_len"]] & 0x02:     # type 8 record: heap id, message flags, ...
                            continue
                        self._attribute(self._heap_object(heap, rec), obj["attrs"])
        return obj

    @staticmethod
    def _undef_bytes(x: bytes) -> bool:
        return x == b"\xff" * len(x)

    def _dataspace(self, m: bytes):
        ver, rank, fl = m[0], m[1], m[2]
        if ver == 1:
            p = 8
        elif ver == 2:
            if m[3] == 2:                           # null dataspace
                return (0,), None
            p = 4
        else:
            self._fail("dataspace version")
        L = self._L
        shape = tuple(int.from_bytes(m[p + i * L:p + (i + 1) * L], "little") for i in range(rank))
        maxshape = None
        if fl & 1:
            p += rank * L
            maxshape = tuple(int.from_bytes(m[p + i * L:p + (i + 1) * L], "little") for i in range(rank))
        return shape, maxshape

    @staticmethod
    def _fillvalue(m: bytes):
        ver = m[0]
        if ver in (1, 2):
            if ver == 2 and not m[3]:
                return None
            n = struct.unpack_from("<I", m, 4)[0]
            return m[8:8 + n] if n else None
        if ver == 3:
            if not m[1] & 0x20:
                return None
            n = struct.unpack_from("<I", m, 2)[0]
            return m[6:6 + n] if n else None
        return None

    @staticmethod
    def _filters(m: bytes):
        ver, n = m[0], m[1]
        out = []
        p = 8 if ver == 1 else 2
        for _ in range(n):
            fid = struct.unpack_from("<H", m, p)[0]
            if ver == 1 or fid >= 256:
                nlen = struct.unpack_from("<H", m, p + 2)[0]
                p += 4
            else:
                nlen = 0
                p += 2
            flags, ncd = struct.unpack_from("<HH", m, p)
            p += 4
            if ver == 1:
                nlen = (nlen + 7) // 8 * 8
            p += nlen
            cd = struct.unpack_from(f"<{ncd}I", m, p)
            p += 4 * ncd
            if ver == 1 and ncd % 2:
                p += 4
            out.append((fid, flags, cd))
        return out

    def _link(self, m: bytes, links: dict):
        fl = m[1]
        p = 2
        ltype = 0
        if fl & 0x08:
            ltype = m[p]
            p += 1
        if fl & 0x04:
            p += 8
        if fl & 0x10:
            p += 1
        n = 1 << (fl & 3)
        nlen = int.from_bytes(m[p:p + n], "little")
        p += n
        name = m[p:p + nlen].decode("utf-8", "replace")
        p += nlen
        if ltype == 0:
            links[name] = int.from_bytes(m[p:p + self._O], "little") + self._base

    def _symbol_table(self, bt: int, heap: int, links: dict):
        b = self._b
        if b[heap:heap + 4] != b"HEAP":
            self._fail("local heap")
        data = self._addr(heap + 8 + 2 * self._L)
        O = self._O

        def walk(node):
            if b[node:node + 4] == b"SNOD":
                n = self._u(node + 6, 2)
                p = node + 8
                for _ in range(n):
                    noff = self._u(p, O)
                    addr = self._u(p + O, O) + self._base
                    s = data + noff
                    e = b.find(b"\x00", s)
                    links[bytes(b[s:e]).decode("utf-8", "replace")] = addr
                    p += 2 * O + 24
                return
            if b[node:node + 4] != b"TREE":
                self._fail("group B-tree")
            n = self._u(node + 6, 2)
            p = node + 8 + 2 * O
            for i in range(n):
                p += self._L                        # key i
                walk(self._u(p, O) + self._base)
                p += O

        walk(bt)

    # ------------------------------------------------------------------ attributes
    def _attribute(self, m: bytes, attrs: dict):
        ver = m[0]
        fl = m[1] if ver >= 2 else 0
        nsz, tsz, ssz = struct.unpack_from("<HHH", m, 2)
        p = 8 + (1 if ver == 3 else 0)
        pad = (lambda n: (n + 7) // 8 * 8) if ver == 1 else (lambda n: n)
        name = m[p:p + nsz].split(b"\x00")[0].decode("utf-8", "replace")
        p += pad(nsz)
        if fl & 0x03:                               # shared datatype / dataspace: user-defined types
            return
        tbuf = m[p:p + tsz]
        p += pad(tsz)
        sbuf = m[p:p + ssz]
        p += pad(ssz)
        try:
            dt = _Datatype(tbuf)
        except NotImplementedError:
            return
        shape, _ = self._dataspace(sbuf) if sbuf else ((), None)
        count = int(np.prod(shape, dtype=np.int64)) if shape else 1
        attrs[name] = self._decode(dt, m[p:], count, shape, attribute=True)

    def _decode(self, dt: _Datatype, raw: bytes, count: int, shape, attribute=False):
        if dt.cls == 9:
            out = []
            step = 4 + self._O + 4
            for i in range(count):
                e = raw[i * step:(i + 1) * step]
                n = struct.unpack_from("<I", e, 0)[0]
                coll = int.from_bytes(e[4:4 + self._O], "little")
                idx = struct.unpack_from("<I", e, 4 + self._O)[0]
                data = self._global_heap(coll + self._base, idx) if n and coll else b""
                if dt.is_vlen_string:
                    out.append(data[:n].decode("utf-8", "replace"))
                else:
                    out.append(np.frombuffer(data[:n * dt.base.size], dtype=dt.base.dtype).copy())
            if dt.is_vlen_string and attribute and not shape:
                return out[0]
            return out
        a = np.frombuffer(raw[:count * dt.size], dtype=dt.dtype)
        if dt.cls == 3:
            vals = [x.split(b"\x00")[0].decode("utf-8", "replace") for x in a.tolist()]
            return vals[0] if attribute and count == 1 else vals
        a = a.astype(dt.dtype.newbyteorder("="))
        if attribute:
            return a[0] if count == 1 else a       # as netCDF4-python: one-element attributes are scalars
        return a.reshape(shape)

    def _global_heap(self, coll: int, idx: int) -> bytes:
        if coll not in self._gcol:
            b = self._b
            if b[coll:coll + 4] != b"GCOL":
                self._fail("global heap")
            size = self._u(coll + 8, self._L)
            objs = {}
            p = coll + 8 + self._L
            end = coll + size
            while p + 8 + self._L <= end:
                i = self._u(p, 2)
                n = self._u(p + 8, self._L)
                if i == 0:
                    break
                objs[i] = bytes(b[p + 8 + self._L:p + 8 + self._L + n])
                p += 8 + self._L + (n + 7) // 8 * 8
            self._gcol[coll] = objs
        return self._gcol[coll].get(idx, b"")

    # ------------------------------------------------------------------ fractal heap + B-tree v2
    def _heap(self, addr: int) -> dict:
        key = ("heap", addr)
        if key in self._objs:
            return self._objs[key]
        b = self._b
        if b[addr:addr + 4] != b"FRHP":
            self._fail("fractal heap")
        O, L = self._O, self._L
        p = addr + 5
        id_len = self._u(p, 2)
        filt_len = self._u(p + 2, 2)
        flags = b[p + 4]
        max_man = self._u(p + 5, 4)
        p += 9
        p += L                                      # next huge id
        huge_bt = None if self._is_undef(p) else self._addr(p)
        p += O
        p += L + O + 4 * L                          # free space, fs manager, managed space, allocated, iterator, #managed
        p += 4 * L                                  # huge size/#, tiny size/#
        width = self._u(p, 2)
        start = self._u(p + 2, L)
        max_direct = self._u(p + 2 + L, L)
        max_heap_bits = self._u(p + 2 + 2 * L, 2)
        p += 2 + 2 * L + 2 + 2                      # ... starting # of rows
        root = None if self._is_undef(p) else self._addr(p)
        cur_rows = self._u(p + O, 2)
        if filt_len:
            raise NotImplementedError("filtered fractal heaps")
        h = {"id_len": id_len, "flags": flags, "width": width, "start": start, "max_direct": max_direct,
             "off_size": (max_heap_bits + 7) // 8, "huge_bt": huge_bt,
             "len_size": min((_log2(max_direct) + 7) // 8, _enc_size(max_man)),
             "max_direct_rows": _log2(max_direct) - _log2(start) + 2, "blocks": []}
        hdr = 5 + O + h["off_size"] + (4 if flags & 2 else 0)

        def row_size(r):
            return start if r < 2 else start << (r - 1)

        def indirect(iaddr, nrows, offset):
            if b[iaddr:iaddr + 4] != b"FHIB":
                self._fail("fractal heap indirect block")
            q = iaddr + 5 + O + h["off_size"]
            for r in range(nrows):
                size = row_size(r)
                for _ in range(width):
                    if r < h["max_direct_rows"]:
                        if not self._is_undef(q):
                            h["blocks"].append((offset, size, self._addr(q)))
                        q += O
                    else:
                        if not self._is_undef(q):
                            indirect(self._addr(q), _log2(size) - _log2(start * width) + 1, offset)
                        q += O
                    offset += size

        if root is not None:
            if cur_rows == 0:
                h["blocks"].append((0, start, root))
            else:
                indirect(root, cur_rows, 0)
        h["hdr"] = hdr
        self._objs[key] = h
        return h

    def _heap_object(self, heap_addr: int, hid: bytes) -> bytes:
        h = self._heap(heap_addr)
        kind = (hid[0] >> 4) & 3
        if kind == 0:                               # managed
            off = int.from_bytes(hid[1:1 + h["off_size"]], "little")
            n = int.from_bytes(hid[1 + h["off_size"]:1 + h["off_size"] + h["len_size"]], "little")
            for boff, bsize, baddr in h["blocks"]:
                if boff <= off < boff + bsize:
                    s = baddr + (off - boff)
                    return bytes(self._b[s:s + n])
            self._fail("fractal heap object outside every block")
        if kind == 2:                               # tiny: the object is in the id
            n = (hid[0] & 0x0F) + 1
            return bytes(hid[1:1 + n])
        # huge
        O, L = self._O, self._L
        if h["id_len"] >= 1 + O + L:
            a = int.from_bytes(hid[1:1 + O], "little") + self._base
            n = int.from_bytes(hid[1 + O:1 + O + L], "little")
            return bytes(self._b[a:a + n])
        want = int.from_bytes(hid[1:1 + L], "little")
        for rec in self._btree2(h["huge_bt"]):      # type 1 record: address, length, id
            if int.from_bytes(rec[O + L:O + 2 * L], "little") == want:
                a = int.from_bytes(rec[:O], "little") + self._base
                n = int.from_bytes(rec[O:O + L], "little")
                return bytes(self._b[a:a + n])
        self._fail("huge fractal heap object not found")

    def _btree2(self, addr: int):
        """All records of a version-2 B-tree, in order."""
        b = self._b
        if b[addr:addr + 4] != b"BTHD":
            self._fail("B-tree v2 header")
        O = self._O
        node_size = self._u(addr + 6, 4)
        rec_size = self._u(addr + 10, 2)
        depth = self._u(addr + 12, 2)
        root = addr + 16
        if self._is_undef(root):
            return []
        nroot = self._u(root + O, 2)
        # per-depth node geometry (H5B2hdr.c)
        max_nrec = [(node_size - 10) // rec_size]
        cum = [max_nrec[0]]
        for d in range(1, depth + 1):
            ptr = O + _enc_size(max_nrec[d - 1]) + (_enc_size(cum[d - 1]) if d > 1 else 0)
            max_nrec.append((node_size - 10 - ptr) // (rec_size + ptr))
            cum.append((max_nrec[d] + 1) * cum[d - 1] + max_nrec[d])
        out = []

        def walk(node, nrec, d):
            sig = b"BTLF" if d == 0 else b"BTIN"
            if b[node:node + 4] != sig:
                self._fail("B-tree v2 node")
            p = node + 6
            recs = [bytes(b[p + i * rec_size:p + (i + 1) * rec_size]) for i in range(nrec)]
            if d == 0:
                out.extend(recs)
                return
            p += nrec * rec_size
            nsz = _enc_size(max_nrec[d - 1])
            tsz = _enc_size(cum[d - 1]) if d > 1 else 0
            for i in range(nrec + 1):
                child = self._addr(p)
                cn = self._u(p + O, nsz)
                p += O + nsz + tsz
                walk(child, cn, d - 1)
                if i < nrec:
                    out.append(recs[i])

        walk(self._addr(root), nroot, depth)
        return out

    # ------------------------------------------------------------------ data
    def _read_dataset(self, obj: dict) -> np.ndarray:
        if obj.get("dtype_error"):
            raise NotImplementedError(obj["dtype_error"])
        dt: _Datatype = obj["dtype"]
        shape = tuple(obj["shape"] or ())
        count = int(np.prod(shape, dtype=np.int64)) if shape else 1
        m = obj["layout"]
        if m is None:
            self._fail("dataset without a layout message")
        ver, cls = m[0], m[1]
        O, L = self._O, self._L
        if dt.cls == 9:
            esize = 4 + O + 4
            ndt = np.dtype(f"V{esize}")
        else:
            esize = dt.size
            ndt = dt.dtype
        fill = obj["fill"]

        def filled(n):
            a = np.zeros(n, dtype=ndt)
            if fill is not None and len(fill) == esize and dt.cls != 9:
                a[:] = np.frombuffer(fill, dtype=ndt)[0]
            return a

        if ver not in (3, 4):
            raise NotImplementedError(f"HDF5 data layout version {ver}")
        if cls == 0:
            n = struct.unpack_from("<H", m, 2)[0]
            flat = np.frombuffer(m[4:4 + n], dtype=ndt)[:count]
        elif cls == 1:
            if self._undef_bytes(m[2:2 + O]):
                flat = filled(count)
            else:
                a = int.from_bytes(m[2:2 + O], "little") + self._base
                flat = np.frombuffer(self._b, dtype=ndt, count=count, offset=a).copy()    # not a view of the map
        elif cls == 2:
            flat = self._read_chunked(obj, m, ver, shape, ndt, esize, filled)
        else:
            raise NotImplementedError("HDF5 virtual / external storage")
        if dt.cls == 9:
            vals = self._decode(dt, flat.tobytes(), count, shape)
            out = np.empty(count, dtype=object)
            out[:] = vals
            return out.reshape(shape)
        if dt.cls == 3:
            return np.array(flat).reshape(shape)
        return np.ascontiguousarray(flat).astype(ndt.newbyteorder("="), copy=False).reshape(shape)

    def _unfilter(self, raw: bytes, filters, mask: int, esize: int) -> bytes:
        for i in range(len(filters) - 1, -1, -1):
            if mask & (1 << i):
                continue
            fid = filters[i][0]
            if fid == 1:
                raw = zlib.decompress(raw)
            elif fid == 2:
                n = len(raw) // esize
                if esize > 1 and n > 0:
                    body = np.frombuffer(raw, dtype=np.uint8, count=n * esize).reshape(esize, n).T.tobytes()
                    raw = body + raw[n * esize:]
            elif fid == 3:
                raw = raw[:-4]
            else:
                raise NotImplementedError(f"HDF5 filter {fid} (only deflate, shuffle and fletcher32 are read)")
        return raw

    def _read_chunked(self, obj, m, ver, shape, ndt, esize, filled):
        b = self._b
        O = self._O
        rank = len(shape)
        if ver == 3:
            nd = m[2]
            bt = None if self._undef_bytes(m[3:3 + O]) else int.from_bytes(m[3:3 + O], "little") + self._base
            cdims = struct.unpack_from(f"<{nd}I", m, 3 + O)[:rank]
            index = "btree1"
        else:
            fl, nd, enc = m[2], m[3], m[4]
            cdims = tuple(int.from_bytes(m[5 + i * enc:5 + (i + 1) * enc], "little") for i in range(nd))[:rank]
            p = 5 + nd * enc
            itype = m[p]
            p += 1
            single = None
            if itype == 1:
                index = "single"
                if fl & 2:
                    single = (int.from_bytes(m[p:p + self._L], "little"), struct.unpack_from("<I", m, p + self._L)[0])
                    p += self._L + 4
            elif itype == 2:
                index = "implicit"
            else:
                raise NotImplementedError("HDF5 1.10 chunk indexes (fixed/extensible array, B-tree v2); "
                                          "the netCDF library does not write them")
            bt = None if self._undef_bytes(m[p:p + O]) else int.from_bytes(m[p:p + O], "little") + self._base
        if nd != rank + 1:
            self._fail("chunk dimensionality")
        out = filled(int(np.prod(shape, dtype=np.int64))).reshape(shape)
        if bt is None or out.size == 0:
            return out.reshape(-1)
        filters = obj["filters"]
        cn = int(np.prod(cdims, dtype=np.int64))

        def place(offs, raw, mask):
            if filters:
                raw = self._unfilter(raw, filters, mask, esize)
            c = np.frombuffer(raw, dtype=ndt, count=cn).reshape(cdims)
            sl = tuple(slice(o, min(o + c_, s)) for o, c_, s in zip(offs, cdims, shape))
            if any(s.start >= s.stop for s in sl):
                return
            out[sl] = c[tuple(slice(0, s.stop - s.start) for s in sl)]

        if index == "single":
            n, mask = single if single else (cn * esize, 0)
            place((0,) * rank, bytes(b[bt:bt + n]), mask)
        elif index == "implicit":
            grid = [(-(-s // c)) for s, c in zip(shape, cdims)]
            for i, idx in enumerate(np.ndindex(*grid)):
                a = bt + i * cn * esize
                place(tuple(k * c for k, c in zip(idx, cdims)), bytes(b[a:a + cn * esize]), 0)
        else:
            ksize = 8 + 8 * nd

            def walk(node):
                if b[node:node + 4] != b"TREE" or b[node + 4] != 1:
                    self._fail("chunk B-tree")
                level = b[node + 5]
                n = self._u(node + 6, 2)
                p = node + 8 + 2 * O
                for _ in range(n):
                    csize, mask = struct.unpack_from("<II", b, p)
                    offs = struct.unpack_from(f"<{rank}Q", b, p + 8)
                    child = self._addr(p + ksize)
                    if level:
                        walk(child)
                    else:
                        place(offs, bytes(b[child:child + csize]), mask)
                    p += ksize + O

            walk(bt)
        return out.reshape(-1)

    # ------------------------------------------------------------------ the netCDF-4 view of the root group
    def _netcdf_view(self, root: dict):
        datasets = {}
        self.groups = []
        for name, addr in root["links"].items():
            o = self._object(addr)
            if o["is_group"] and o["layout"] is None:
                self.groups.append(name)
            elif o["shape"] is not None and (o["dtype"] is not None or o.get("dtype_error")):
                datasets[name] = o
        # dimensions = dimension scales, ordered by _Netcdf4Dimid when present
        scales = []
        for name, o in datasets.items():
            cls = o["attrs"].get("CLASS")
            if isinstance(cls, str) and cls == "DIMENSION_SCALE":
                dimid = o["attrs"].get("_Netcdf4Dimid")
                scales.append((int(dimid) if dimid is not None else len(scales) + (1 << 20), name, o))
        scales.sort(key=lambda t: t[0])
        self.dimensions = {}
        self.unlimited = set()
        by_addr, by_id = {}, {}
        for dimid, name, o in scales:
            dname = name[len("_nc4_non_coord_"):] if name.startswith("_nc4_non_coord_") else name
            self.dimensions[dname] = int(o["shape"][0]) if o["shape"] else 1
            if o["maxshape"] and o["maxshape"][0] == _UNDEF[8]:
                self.unlimited.add(dname)
            by_addr[o["addr"]] = dname
            by_id[dimid] = dname
        self.variables = {}
        phony = {}
        for name, o in datasets.items():
            nm = o["attrs"].get("NAME")
            if isinstance(nm, str) and nm.startswith(_NOT_A_VAR):
                continue
            vname = name[len("_nc4_non_coord_"):] if name.startswith("_nc4_non_coord_") else name
            if o["dtype"] is None:
                continue                            # user-defined type: not exposed
            v = Variable(self, vname, o)
            rank = len(v.shape)
            dl = o["attrs"].get("DIMENSION_LIST")
            coords = o["attrs"].get("_Netcdf4Coordinates")
            dims = None
            if rank == 0:
                dims = ()
            elif dl is not None and len(dl) == rank and all(len(x) and int(x[0]) + self._base in by_addr for x in dl):
                dims = tuple(by_addr[int(x[0]) + self._base] for x in dl)
            elif coords is not None and len(np.atleast_1d(coords)) == rank and \
                    all(int(c) in by_id for c in np.atleast_1d(coords)):
                dims = tuple(by_id[int(c)] for c in np.atleast_1d(coords))
            elif o["addr"] in by_addr and rank == 1:
                dims = (by_addr[o["addr"]],)
            else:                                   # plain HDF5 without scales: phony dimensions by size
                dims = []
                for n in v.shape:
                    dims.append(phony.setdefault(n, f"phony_dim_{len(phony)}"))
                    self.dimensions.setdefault(dims[-1], int(n))
                dims = tuple(dims)
            v.dims = dims
            self.variables[vname] = v

    def __repr__(self):
        return f"<nc4.File {self.path}: {len(self.variables)} variables, dims {self.dimensions}>"
