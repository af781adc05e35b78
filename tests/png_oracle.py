"""NumPy restatement of the library's PNG encoding (include/vsc_b200.h, VSC_ENCODE_PNG): the row filter exactly, a
checker for any file that claims to encode a frame with it, and the size of the zlib Z_RLE model it is measured against."""
import struct
import zlib

import numpy as np

SEG = 32768                      # filtered-stream bytes per deflate segment
SIG = b'\x89PNG\r\n\x1a\n'


def _paeth(a, b, c):
    p = a + b - c
    pa, pb, pc = np.abs(p - a), np.abs(p - b), np.abs(p - c)
    return np.where((pa <= pb) & (pa <= pc), a, np.where(pb <= pc, b, c))


def _candidates(frame):
    """The five filtered forms of every row, [5, h, 3w] int32 in 0..255."""
    h, w, _ = frame.shape
    x = frame.reshape(h, 3 * w).astype(np.int32)
    up = np.vstack([np.zeros((1, 3 * w), np.int32), x[:-1]])
    left = np.hstack([np.zeros((h, 3), np.int32), x[:, :-3]])
    ul = np.hstack([np.zeros((h, 3), np.int32), up[:, :-3]])
    return np.stack([x, x - left, x - up, x - (left + up) // 2, x - _paeth(left, up, ul)]) & 255


def filter_rows(frame: np.ndarray) -> bytes:
    """The filtered stream of an rgb24 frame [h, w, 3]: per row the filter type byte, then the row filtered with the type
    of least sum(min(b, 256 - b)) (ties: the lowest type; row 0 against a zero row)."""
    frame = np.ascontiguousarray(frame, np.uint8)
    parts = []
    for y0 in range(0, frame.shape[0], 64):                 # blocks of rows (with the row above) bound the memory
        lo = max(y0 - 1, 0)
        f = _candidates(frame[lo:y0 + 64])[:, y0 - lo:]
        cost = np.minimum(f, 256 - f).sum(axis=2)            # [5, rows]
        t = np.argmin(cost, axis=0)                           # first minimum = lowest type
        rows = f[t, np.arange(f.shape[1])]
        parts.append(np.hstack([t[:, None], rows]).astype(np.uint8).tobytes())
    return b''.join(parts)


def unfilter(data: bytes, h: int, w: int) -> np.ndarray:
    """Inverse of filter_rows (any filter types): the rgb24 frame [h, w, 3]."""
    rb = 3 * w
    a = np.frombuffer(data, np.uint8).reshape(h, rb + 1)
    out = np.zeros((h, rb), np.int32)
    prev = np.zeros(rb, np.int32)
    for y in range(h):
        t, row = int(a[y, 0]), a[y, 1:].astype(np.int32)
        cur = np.zeros(rb, np.int32)
        if t in (0, 2):
            cur = (row + (prev if t == 2 else 0)) & 255
        else:
            for i in range(rb):
                left = cur[i - 3] if i >= 3 else 0
                ul = prev[i - 3] if i >= 3 else 0
                pred = left if t == 1 else (left + prev[i]) // 2 if t == 3 else int(_paeth(np.int32(left), np.int32(prev[i]), np.int32(ul)))
                cur[i] = (row[i] + pred) & 255
        out[y] = cur
        prev = cur
    return out.astype(np.uint8).reshape(h, w, 3)


def chunks(data: bytes):
    """[(type, payload)] of a PNG file; asserts the signature, every chunk CRC and that nothing trails IEND."""
    assert data[:8] == SIG, 'PNG signature'
    out, pos = [], 8
    while pos < len(data):
        n, = struct.unpack('>I', data[pos:pos + 4])
        typ, body = data[pos + 4:pos + 8], data[pos + 8:pos + 8 + n]
        crc, = struct.unpack('>I', data[pos + 8 + n:pos + 12 + n])
        assert crc == zlib.crc32(typ + body), f'CRC of chunk {len(out)} ({typ!r})'
        out.append((typ, body))
        pos += 12 + n
        if typ == b'IEND':
            break
    assert pos == len(data), 'bytes after IEND'
    return out


def check_png(data, frame: np.ndarray) -> None:
    """Assert that `data` is the library's PNG file of the rgb24 frame [h, w, 3]: chunk set, CRCs, IHDR, zlib header, one
    IDAT per segment, a zlib stream (Adler-32 included) inflating to exactly filter_rows(frame), and a cv2 decode to
    the frame."""
    import cv2
    data = bytes(data)
    h, w, _ = frame.shape
    cs = chunks(data)
    assert cs[0] == (b'IHDR', struct.pack('>IIBBBBB', w, h, 8, 2, 0, 0, 0)), 'IHDR'
    assert cs[-1] == (b'IEND', b'')
    idat = [c for c in cs[1:-1]]
    assert all(t == b'IDAT' for t, _ in idat)
    filtered = filter_rows(frame)
    assert len(idat) == -(-len(filtered) // SEG), 'one IDAT per segment'
    z = b''.join(b for _, b in idat)
    assert z[:2] == b'\x78\x01', 'zlib header'
    assert z[-10:-4] == b'\x00\x00\xff\xff\x03\x00', 'sync flush, then the final empty fixed block'
    d = zlib.decompressobj()
    raw = d.decompress(z)
    assert d.eof and not d.unused_data, 'zlib stream ends with the Adler-32'
    assert raw == filtered, 'inflated stream is the filtered stream'
    img = cv2.imdecode(np.frombuffer(data, np.uint8), cv2.IMREAD_UNCHANGED)
    assert img is not None and img.shape == frame.shape and np.array_equal(img[..., ::-1], frame), 'cv2 decode'


def assemble(frame: np.ndarray) -> bytes:
    """A PNG file of the frame built with zlib from filter_rows (the reference the format's framing is checked against)."""
    h, w, _ = frame.shape

    def chunk(t, b):
        return struct.pack('>I', len(b)) + t + b + struct.pack('>I', zlib.crc32(t + b))
    return (SIG + chunk(b'IHDR', struct.pack('>IIBBBBB', w, h, 8, 2, 0, 0, 0)) + chunk(b'IDAT', zlib.compress(filter_rows(frame)))
            + chunk(b'IEND', b''))


def model_size(frame: np.ndarray, seg: int = SEG) -> int:
    """Bytes of the zlib model of the format: filter_rows, then zlib Z_RLE on every segment on its own, sync-flushed, in
    the library's framing (signature, IHDR, one IDAT per segment, zlib header, final block, Adler-32, IEND)."""
    f = filter_rows(frame)
    body = 0
    for o in range(0, len(f), seg):
        c = zlib.compressobj(6, zlib.DEFLATED, -15, 8, zlib.Z_RLE)
        body += len(c.compress(f[o:o + seg]) + c.flush(zlib.Z_SYNC_FLUSH))
    nseg = -(-len(f) // seg)
    return 8 + 25 + 12 * nseg + 2 + body + 2 + 4 + 12
