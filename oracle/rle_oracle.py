"""COCO compressed RLE, restated from pycocotools' common/maskApi.c (the file behind pycocotools.mask.encode / decode /
area / toBbox).  Each step quotes the C statement it restates.  pycocotools is not installed here, so parity with the
package itself is not pinned by a run; the hand-checked strings of tests/test_rle_oracle_cpu.py are.

  encode(mask)          rleEncode over the Fortran (column-major) order of an [h, w] 0/1 mask -> counts (int64)
  to_string(counts)     rleToString -> bytes
  fr_string(s)          rleFrString -> counts
  decode(counts, h, w)  rleDecode -> uint8 [h, w]
  area(counts)          rleArea
  to_bbox(counts, h, w) rleToBbox -> float64 [x, y, w, h]
  encode_mask(mask)     pycocotools.mask.encode's dict {'size': [h, w], 'counts': bytes}, with area and bbox
  CEncoder              the single-threaded C restatement of rleEncode + rleToString (rle_oracle.c, compiled on
                        first use into the temporary directory)
"""
import ctypes as C
import hashlib
import os
import shutil
import subprocess
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))


def encode(mask):
    """rleEncode: `for(j=0; j<a; j++) { if(T[j]!=p) { cnts[k++]=c; c=0; p=T[j]; } c++; } cnts[k++]=c;` with p = 0,
    c = 0 and T the mask in column-major order (pixel j = x*h + y).  The counts are the distances between the
    positions where T differs from the pixel before it (a virtual 0 precedes pixel 0), then the rest to a = h*w."""
    t = np.asarray(mask).T.reshape(-1) != 0                  # T[j], j = x*h + y
    prev = np.concatenate(([False], t[:-1]))
    pos = np.flatnonzero(t != prev)                          # every j with T[j] != p
    return np.diff(np.concatenate(([0], pos, [t.size]))).astype(np.int64)


def to_string(cnts):
    """rleToString: for each count i, `x=(long) cnts[i]; if(i>2) x-=(long) cnts[i-2]; more=1; while( more ) {
    char c=x & 0x1f; x >>= 5; more=(c & 0x10) ? x!=-1 : x!=0; if(more) c |= 0x20; c+=48; s[p++]=c; }`.
    The while loop runs for all counts at once: round k emits the k-th character of every count still going."""
    cnts = np.asarray(cnts, dtype=np.int64)
    x = cnts.copy()
    x[3:] -= cnts[1:-2]                                      # i > 2 (not i >= 2)
    going = np.ones(x.size, bool)
    rounds = []
    for _ in range(7):                                       # a 32-bit count takes at most 7 characters
        c = x & 0x1f
        x = x >> 5                                           # arithmetic shift of a signed 64-bit value
        more = np.where(c & 0x10, x != -1, x != 0)
        rounds.append(np.where(going, (c | np.where(more, 0x20, 0)) + 48, -1))
        going &= more
    assert not going.any()
    chars = np.stack(rounds, 1).reshape(-1)                  # count-major, character order within a count
    return chars[chars >= 0].astype(np.uint8).tobytes()


def fr_string(s):
    """rleFrString: `while( s[p] ) { x=0; k=0; more=1; while( more ) { c=s[p]-48; x |= (c & 0x1f) << 5*k;
    more = c & 0x20; p++; k++; if(!more && (c & 0x10)) x |= -1 << 5*k; } if(m>2) x+=(long) cnts[m-2];
    cnts[m++]=(uint) x; }`."""
    cnts, p = [], 0
    while p < len(s):
        x, k, more = 0, 0, True
        while more:
            c = s[p] - 48
            x |= (c & 0x1f) << (5 * k)
            more = c & 0x20
            p += 1
            k += 1
            if not more and (c & 0x10):
                x |= -1 << (5 * k)
        if len(cnts) > 2:
            x += cnts[-2]
        cnts.append(x & 0xffffffff)                          # (uint) x
    return np.array(cnts, dtype=np.int64)


def decode(cnts, h, w):
    """rleDecode: `v=0; for( j=0; j<R[i].m; j++ ) { for( k=0; k<R[i].cnts[j]; k++ ) *(M++)=v; v=!v; }`, Fortran
    order back to [h, w]."""
    cnts = np.asarray(cnts, dtype=np.int64)
    vals = np.arange(cnts.size) % 2
    return np.repeat(vals, cnts).astype(np.uint8).reshape(w, h).T


def area(cnts):
    """rleArea: `a[i]=0; for( j=1; j<R[i].m; j+=2 ) a[i]+=R[i].cnts[j];`."""
    return int(np.asarray(cnts, dtype=np.int64)[1::2].sum())


def to_bbox(cnts, h, w):
    """rleToBbox: `m=((siz)(m/2))*2; xs=w; ys=h; xe=ye=0; cc=0; if(m==0) { bb = 0 } for( j=0; j<m; j++ ) {
    cc+=R[i].cnts[j]; t=cc-j%2; y=t%h; x=(t-y)/h; if(j%2==0) xp=x; else if(xp<x) { ys=0; ye=h-1; }
    xs=umin(xs,x); xe=umax(xe,x); ys=umin(ys,y); ye=umax(ye,y); } bb = [xs, ys, xe-xs+1, ye-ys+1]`."""
    cnts = np.asarray(cnts, dtype=np.int64)
    m = (cnts.size // 2) * 2
    if m == 0:
        return np.zeros(4, np.float64)
    j = np.arange(m)
    t = np.cumsum(cnts[:m]) - j % 2                          # first pixel of each run of ones, last pixel of it
    y, x = t % h, t // h
    xs, xe, ys, ye = x.min(), x.max(), y.min(), y.max()
    if np.any(x[0::2] < x[1::2]):                            # a run across a column boundary
        ys, ye = 0, h - 1
    return np.array([xs, ys, xe - xs + 1, ye - ys + 1], np.float64)


def encode_mask(mask):
    """pycocotools.mask.encode(np.asfortranarray(mask)) for one [h, w] mask, with mask.area and mask.toBbox:
    ({'size': [h, w], 'counts': bytes}, area, bbox float64 [4])."""
    h, w = np.asarray(mask).shape
    cnts = encode(mask)
    return {"size": [h, w], "counts": to_string(cnts)}, area(cnts), to_bbox(cnts, h, w)


_cpu = None


def _lib():
    """rle_oracle.c compiled on first use into the temporary directory (the tree may be read-only), keyed by the
    source's hash so that an edited source is rebuilt."""
    global _cpu
    if _cpu is None:
        src = os.path.join(HERE, "rle_oracle.c")
        with open(src, "rb") as f:
            key = hashlib.sha256(f.read()).hexdigest()[:16]
        path = os.path.join(tempfile.gettempdir(), f"cim_rle_oracle_{os.getuid()}_{key}.so")
        if not os.path.exists(path):
            fd, tmp = tempfile.mkstemp(suffix=".so", dir=os.path.dirname(path))
            os.close(fd)
            try:
                cc = next(filter(None, map(shutil.which, (os.environ.get("CC", ""), "cc", "gcc", "clang"))), None)
                if cc is None:
                    raise RuntimeError("no C compiler (CC, cc, gcc or clang) to build oracle/rle_oracle.c")
                subprocess.run([cc, "-O2", "-fPIC", "-shared", "-o", tmp, src], check=True)
                os.replace(tmp, path)                        # atomic: concurrent first uses do not see half a file
            finally:
                if os.path.exists(tmp):
                    os.remove(tmp)
        lib = C.CDLL(path)
        lib.rle_oracle_encode.restype = C.c_int64
        lib.rle_oracle_encode.argtypes = [C.c_void_p, C.c_int64, C.c_int64, C.c_void_p, C.c_void_p, C.c_int64]
        _cpu = lib
    return _cpu


class CEncoder:
    """The C restatement of rleEncode + rleToString (oracle/rle_oracle.c), one mask at a time on one thread, over
    uint8 masks in Fortran order (np.asfortranarray(mask), what pycocotools.mask.encode takes).  Scratch buffers are
    allocated once for masks of up to h*w pixels."""

    def __init__(self, hw):
        self.cnts = np.empty(hw + 1, np.uint32)
        self.chars = np.empty(7 * (hw + 1), np.uint8)
        self.lib = _lib()

    def __call__(self, mask_f):
        assert mask_f.dtype == np.uint8 and mask_f.flags.f_contiguous and mask_f.size < self.cnts.size
        h, w = mask_f.shape
        n = self.lib.rle_oracle_encode(mask_f.ctypes.data, h, w, self.cnts.ctypes.data, self.chars.ctypes.data,
                                       self.chars.size)
        return self.chars[:n].tobytes()
