"""brpc::policy::GzipDecompress(const IOBuf&, IOBuf*) = GzipDecompressBase (src/brpc/policy/gzip_compress.cpp:138-176) restated on the
system zlib (tests only): protobuf's GzipInputStream with Next() as a method, driven the way GzipDecompressBase drives it, over a body
in ONE block.  It is the pin of orc_h2_decompress (oracle/b2_oracle_h2_gzip.c) and, through it, of b2_h2_decompress_requests.  The zlib
calls are tests/_gzipstream.py's."""
import ctypes as C

from _gzipstream import GZIP, K_BUFFER, Z_BUF_ERROR, Z_NO_FLUSH, Z_OK, Z_STREAM_END, ZStream, _init, _z


class GzipInputStream:
    """GzipInputStream(sub_stream = one IOBuf block holding `data`, GZIP) with Next() as a method, for callers that drive it
    themselves.  sub_byte_count is the sub-stream's ByteCount() (the block once Next() took it; nothing is ever backed up)."""

    def __init__(self, data: bytes, fmt: int = GZIP):
        self.data, self.fmt = data, fmt
        self.zs = ZStream()
        self.src = C.create_string_buffer(data, len(data)) if data else C.create_string_buffer(1)
        self.outbuf = C.create_string_buffer(K_BUFFER)
        self.out_base = C.addressof(self.outbuf)
        self.zs.next_out = self.out_base; self.zs.avail_out = K_BUFFER
        self.output_position = self.out_base
        self.zerror = Z_OK
        self.sub_used = False
        self.sub_byte_count = 0

    def _sub_next(self):
        if self.sub_used or len(self.data) == 0:        # IOBufAsZeroCopyInputStream: an empty IOBuf has no block
            return False
        self.sub_used = True; self.sub_byte_count = len(self.data)
        return True

    def _inflate(self):
        zs = self.zs
        if self.zerror == Z_OK and zs.avail_out == 0:
            pass
        elif zs.avail_in == 0:
            first = not zs.next_in
            if not self._sub_next():
                zs.next_out = None; zs.avail_out = 0
                return Z_STREAM_END
            zs.next_in = C.addressof(self.src); zs.avail_in = len(self.data)
            if first:
                e = _init(zs, self.fmt)
                if e != Z_OK:
                    return e
        zs.next_out = self.out_base; zs.avail_out = K_BUFFER
        self.output_position = self.out_base
        return _z.inflate(C.byref(zs), Z_NO_FLUSH)

    def _do_next_output(self):
        n = (self.zs.next_out or 0) - self.output_position
        b = C.string_at(self.output_position, n)
        self.output_position = self.zs.next_out
        return b

    def next(self):
        """Next(): the bytes handed over, or None for false."""
        zs = self.zs
        if self.zerror not in (Z_OK, Z_STREAM_END, Z_BUF_ERROR) or not zs.next_out:
            return None
        if zs.next_out != self.output_position:
            return self._do_next_output()
        if self.zerror == Z_STREAM_END:
            self.zerror = _z.inflateEnd(C.byref(zs))
            if self.zerror != Z_OK:
                return None
            self.zerror = _init(zs, self.fmt)
            if self.zerror != Z_OK:
                return None
        self.zerror = self._inflate()
        if self.zerror == Z_STREAM_END and not zs.next_out:
            return None
        if self.zerror not in (Z_OK, Z_STREAM_END, Z_BUF_ERROR):
            return None
        return self._do_next_output()

    def close(self):
        if self.zs.state:
            _z.inflateEnd(C.byref(self.zs))
            self.zs.state = None


def gzip_decompress_base(data: bytes):
    """brpc::policy::GzipDecompress(const IOBuf&, IOBuf*) = GzipDecompressBase (gzip_compress.cpp:138-176) over a body in one
    block, call for call: copy out what Next() hands over; false when the sub-stream was not read to its end or when one more
    Next() succeeds.  Returns (ok, bytes)."""
    s = GzipInputStream(data, GZIP)
    got = bytearray()
    try:
        size_in = 0
        while True:                                     # out.Next() of an IOBufAsZeroCopyOutputStream always succeeds
            if size_in == 0:
                b = s.next()
                if b is None:
                    break
                size_in = len(b)
                got.extend(b)
            size_in = 0                                 # (memcpy of min(size_in, size_out) in block-sized steps: all of it)
        ok = not (size_in != 0 or s.sub_byte_count != len(data) or s.next() is not None)
    finally:
        s.close()
    return ok, bytes(got)
