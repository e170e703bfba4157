"""Call-by-call driver of a library with the zlib.h ABI: the same script of deflate() / inflate() calls and their
companions runs on libzb200.so and on the system zlib, and every call is recorded -- return code, input consumed,
output produced (the bytes), total_in, total_out, adler, msg -- so that two libraries can be compared call for call.
binding.z_stream is the 112-byte LP64 layout of both, and zlib 1.2.x and 1.3 both accept binding.ZLIB_VERSION.
Test infrastructure only."""
import ctypes as C
import os
from collections import namedtuple

from zlib_b200 import binding as zb

NAMES = ("deflateInit2_", "deflate", "deflateEnd", "deflateReset", "deflateCopy", "deflateParams", "deflatePrime",
         "deflateSetDictionary", "deflateSetHeader", "deflateBound",
         "inflateInit2_", "inflate", "inflateEnd", "inflateReset", "inflateCopy", "inflateSync", "inflateSetDictionary",
         "inflateGetHeader", "inflatePrime")

SYSTEM_ZLIB = ("/lib/x86_64-linux-gnu/libz.so.1", "/usr/lib/x86_64-linux-gnu/libz.so.1")    # as test_multi_gpu finds it


def system_zlib_path():
    for p in SYSTEM_ZLIB:
        if os.path.exists(p):
            return p
    return None


class Api:
    """The zlib.h entry points of one library, typed by binding's table (libzb200.so already is)."""

    def __init__(self, dll, name):
        sigs = zb.signatures()
        for n in NAMES:
            f = getattr(dll, n)
            f.restype, f.argtypes = sigs[n]
        self.dll, self.name = dll, name


def system_zlib():
    p = system_zlib_path()
    return Api(C.CDLL(p, mode=os.RTLD_LOCAL | os.RTLD_DEEPBIND), "zlib") if p else None


# one call: op, return code, input bytes consumed, output bytes, and the stream fields after it; avail_in is what the
# caller still holds (input handed over and not consumed), avail_out the room left
Rec = namedtuple("Rec", "op rc used out total_in total_out adler msg avail_in avail_out")


class Stream:
    """One z_stream of `api`.  Input handed to a call and not consumed stays queued in front of the next call's piece,
    as a caller that keeps its input buffer does."""

    def __init__(self, api, kind, wbits=15, level=6, mem_level=8, strategy=0, _copy_of=None):
        self.api, self.kind = api, kind
        self.s = zb.z_stream()
        self.pending = b""
        self.keep = []                                          # gz_header and its buffers, alive while the stream is
        self.open = False
        if _copy_of is not None:
            return
        if kind == "inflate":
            rc = api.dll.inflateInit2_(C.byref(self.s), wbits, zb.ZLIB_VERSION, C.sizeof(zb.z_stream))
        else:
            rc = api.dll.deflateInit2_(C.byref(self.s), level, zb.Z_DEFLATED, wbits, mem_level, strategy,
                                       zb.ZLIB_VERSION, C.sizeof(zb.z_stream))
        assert rc == zb.Z_OK, (api.name, kind, wbits, level, mem_level, strategy, rc)
        self.open = True

    def _rec(self, op, rc, used, out):
        s = self.s
        return Rec(op, rc, used, out, s.total_in, s.total_out, s.adler, s.msg.decode() if s.msg else None, len(self.pending),
                   s.avail_out)

    def call(self, op, data=b"", room=0, arg=0):
        """op: "inflate" / "deflate" (arg = flush), "sync", "reset", "params" (arg = (level, strategy)), "prime" (arg =
        (bits, value): deflatePrime or inflatePrime), "dict" (arg = dictionary).  `data` joins the queued input, `room` is avail_out."""
        d, s = self.api.dll, self.s
        self.pending += bytes(data)
        inbuf = C.create_string_buffer(self.pending, len(self.pending) + 1)
        outbuf = C.create_string_buffer(max(room, 1))
        s.next_in, s.avail_in = C.addressof(inbuf), len(self.pending)
        s.next_out, s.avail_out = C.addressof(outbuf), room
        p = C.byref(s)
        if op == "inflate":
            rc = d.inflate(p, arg)
        elif op == "deflate":
            rc = d.deflate(p, arg)
        elif op == "sync":
            rc = d.inflateSync(p)
        elif op == "reset":
            rc = d.inflateReset(p) if self.kind == "inflate" else d.deflateReset(p)
        elif op == "params":
            rc = d.deflateParams(p, *arg)
        elif op == "prime":
            rc = (d.inflatePrime if self.kind == "inflate" else d.deflatePrime)(p, *arg)
        elif op == "dict":
            f = d.inflateSetDictionary if self.kind == "inflate" else d.deflateSetDictionary
            rc = f(p, bytes(arg), len(arg))
        else:
            raise ValueError(op)
        used = len(self.pending) - s.avail_in
        assert 0 <= used <= len(self.pending) and s.next_in == C.addressof(inbuf) + used, (self.api.name, op)
        self.pending = self.pending[used:]
        out = outbuf.raw[:room - s.avail_out]
        return self._rec(op, rc, used, out)

    def set_header(self, text=0, time=0, os_=3, extra=None, name=None, comment=None, hcrc=0):
        """deflateSetHeader with these fields (bytes; name and comment without their zero)."""
        h = zb.gz_header()
        h.text, h.time, h.os, h.hcrc = text, time, os_, hcrc
        bufs = []
        if extra is not None:
            b = C.create_string_buffer(extra, len(extra) + 1)
            h.extra, h.extra_len = C.addressof(b), len(extra)
            bufs.append(b)
        if name is not None:
            b = C.create_string_buffer(name + b"\0")
            h.name = C.addressof(b)
            bufs.append(b)
        if comment is not None:
            b = C.create_string_buffer(comment + b"\0")
            h.comment = C.addressof(b)
            bufs.append(b)
        self.keep += [h] + bufs
        return self.api.dll.deflateSetHeader(C.byref(self.s), C.addressof(h))

    def get_header(self, room=256):
        """inflateGetHeader with `room` bytes for each of extra, name and comment -> the gz_header (filled as it goes)."""
        h = zb.gz_header()
        bufs = [C.create_string_buffer(room) for _ in range(3)]
        h.extra, h.extra_max = C.addressof(bufs[0]), room
        h.name, h.name_max = C.addressof(bufs[1]), room
        h.comment, h.comm_max = C.addressof(bufs[2]), room
        self.keep += [h] + bufs
        assert self.api.dll.inflateGetHeader(C.byref(self.s), C.addressof(h)) == zb.Z_OK
        return h

    def bound(self, n):
        return self.api.dll.deflateBound(C.byref(self.s), n)

    def copy(self):
        """deflateCopy / inflateCopy into a new Stream, which takes the queued input along -> (rc, Stream)."""
        other = Stream(self.api, self.kind, _copy_of=self)
        f = self.api.dll.inflateCopy if self.kind == "inflate" else self.api.dll.deflateCopy
        rc = f(C.byref(other.s), C.byref(self.s))
        other.open = rc == zb.Z_OK
        other.pending = self.pending
        return rc, other

    def close(self):
        if self.open:
            self.open = False
            return (self.api.dll.inflateEnd if self.kind == "inflate" else self.api.dll.deflateEnd)(C.byref(self.s))
        return None

    def __del__(self):
        self.close()


def run(api, kind, script, **init):
    """The records of one script on a fresh stream; a step is (op, data, room, arg)."""
    st = Stream(api, kind, **init)
    try:
        return [st.call(*step) for step in script]
    finally:
        st.close()


def joined(recs):
    return b"".join(r.out for r in recs)


# ---- inflate: this library against zlib, call for call ---------------------------------------------------------------
# zlib's inflate() makes all the progress its input and room allow, and zlib.h asks that of every implementation: so
# output per call is zlib's, and so is the return code -- except that a call whose only progress in zlib was input
# pulled into its bit buffer (no output) may say Z_BUF_ERROR here where zlib says Z_OK.  total_in is zlib's whenever
# the call ended for lack of input (all of it taken, room left) or at the end of the stream, and at Z_NEED_DICT the
# input left behind the dictionary id is zlib's (zlib's total_in leaves out the bytes of that call, for the rest of the
# stream, so from there on only the input left is compared).  Not compared: total_in at
# Z_DATA_ERROR (zlib has pulled the bytes of the bad code into its bit buffer, this library counts up to the code), and
# adler of raw streams (zlib 1.3 leaves 0 there, 1.2.3 and this library 1).
def inflate_mismatch(got, want, raw=False, lag=False):
    """None when record `got` of this library may stand beside zlib's `want`, else what differs."""
    if got.op != want.op:
        return "op %s vs %s" % (got.op, want.op)
    if got.out != want.out:
        n = next((i for i, (a, b) in enumerate(zip(got.out, want.out)) if a != b), min(len(got.out), len(want.out)))
        return "output: %d bytes vs zlib's %d, first difference at %d" % (len(got.out), len(want.out), n)
    if got.rc != want.rc and not (want.rc == zb.Z_OK and got.rc == zb.Z_BUF_ERROR and not want.out
                                  and got.op == "inflate"):
        return "rc %d vs zlib's %d" % (got.rc, want.rc)
    if got.total_out != want.total_out:
        return "total_out %d vs zlib's %d" % (got.total_out, want.total_out)
    ended = want.rc == zb.Z_STREAM_END or (want.rc not in (zb.Z_DATA_ERROR, zb.Z_NEED_DICT) and want.avail_in == 0
                                           and want.avail_out > 0)
    if ended and (got.avail_in, got.total_in if not lag else 0) != (want.avail_in, want.total_in if not lag else 0):
        return "total_in %d, %d left vs zlib's %d, %d left" % (got.total_in, got.avail_in, want.total_in, want.avail_in)
    if want.rc == zb.Z_NEED_DICT and got.avail_in != want.avail_in:     # zlib leaves total_in behind there
        return "%d left vs zlib's %d at Z_NEED_DICT" % (got.avail_in, want.avail_in)
    if want.rc in (zb.Z_STREAM_END, zb.Z_NEED_DICT) and got.adler != want.adler and not raw:
        return "adler %#x vs zlib's %#x" % (got.adler, want.adler)
    if want.rc == zb.Z_DATA_ERROR and got.msg != want.msg:
        return "msg %r vs zlib's %r" % (got.msg, want.msg)
    return None


def inflate_diff(got, want, raw=False):
    """(call index, what differs) of the first call that breaks the rules, or None."""
    if len(got) != len(want):
        return (min(len(got), len(want)), "%d calls vs zlib's %d" % (len(got), len(want)))
    lag = False
    for i, (g, w) in enumerate(zip(got, want)):
        m = inflate_mismatch(g, w, raw, lag)
        if m:
            return (i, m + "  [ours %s | zlib %s]" % (_short(g), _short(w)))
        lag = lag or w.rc == zb.Z_NEED_DICT
    return None


def _short(r):
    return "%s rc=%d used=%d out=%d tin=%d tout=%d left=%d msg=%r" % (r.op, r.rc, r.used, len(r.out), r.total_in,
                                                                      r.total_out, r.avail_in, r.msg)
