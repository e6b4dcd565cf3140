"""GPU tests of the streaming / state API of the zlib ABI (SURVEY.md section 8 row f1): block-resumable inflate(), gz_header on
both sides, dictionaries on the inflate side, inflateSync / SyncPoint / Prime / GetDictionary / Back, and the truncation rules the
advisor asked for.  Everything goes through libz_b200.so's z_stream entry points; stock zlib and the oracle are the checkers."""
import ctypes
import os
import sys
import zlib

import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
sys.path.insert(0, os.path.dirname(HERE))

import zlib_rs_b200 as Z  # noqa: E402
import oracle_lib as O  # noqa: E402
from corpus import silesia_member, silesia_tar, synthetic_mix  # noqa: E402

pytestmark = pytest.mark.gpu

Z_OK, Z_STREAM_END, Z_NEED_DICT, Z_DATA_ERROR, Z_BUF_ERROR, Z_STREAM_ERROR = 0, 1, 2, -3, -5, -2
Z_NO_FLUSH, Z_SYNC_FLUSH, Z_FULL_FLUSH, Z_FINISH = 0, 2, 3, 4


class GzHeader(ctypes.Structure):
    _fields_ = [("text", ctypes.c_int), ("time", ctypes.c_ulong), ("xflags", ctypes.c_int), ("os", ctypes.c_int),
                ("extra", ctypes.c_void_p), ("extra_len", ctypes.c_uint), ("extra_max", ctypes.c_uint),
                ("name", ctypes.c_void_p), ("name_max", ctypes.c_uint), ("comment", ctypes.c_void_p),
                ("comm_max", ctypes.c_uint), ("hcrc", ctypes.c_int), ("done", ctypes.c_int)]


def L():
    lib = Z.lib()
    zs = ctypes.POINTER(Z.ZStream)
    lib.inflateSetDictionary.argtypes = [zs, ctypes.c_void_p, ctypes.c_uint]
    lib.inflateGetDictionary.argtypes = [zs, ctypes.c_void_p, ctypes.POINTER(ctypes.c_uint)]
    lib.inflateGetHeader.argtypes = [zs, ctypes.POINTER(GzHeader)]
    lib.deflateSetHeader.argtypes = [zs, ctypes.POINTER(GzHeader)]
    lib.inflateSync.argtypes = [zs]
    lib.inflateSyncPoint.argtypes = [zs]
    lib.inflatePrime.argtypes = [zs, ctypes.c_int, ctypes.c_int]
    lib.inflateReset.argtypes = [zs]
    lib.inflateReset2.argtypes = [zs, ctypes.c_int]
    lib.inflateValidate.argtypes = [zs, ctypes.c_int]
    lib.inflateMark.argtypes, lib.inflateMark.restype = [zs], ctypes.c_long
    lib.deflateUsed.argtypes = [zs, ctypes.POINTER(ctypes.c_int)]
    lib.deflateTune.argtypes = [zs, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int]
    return lib


class Inf:
    """inflate() driven call by call; keeps the input buffer of the current call alive."""

    def __init__(self, wbits=15):
        self.s = Z.ZStream()
        rc = L().inflateInit2_(ctypes.byref(self.s), wbits, Z.ZLIB_VERSION, ctypes.sizeof(Z.ZStream))
        assert rc == Z_OK, rc
        self.out = bytearray()

    def feed(self, data, flush=Z_NO_FLUSH, out_chunk=1 << 15):
        """One input chunk, inflate() until it stops making output.  Returns the last return code."""
        data = bytes(data)
        src = (ctypes.c_char * max(len(data), 1)).from_buffer_copy(data or b"\0")
        self.s.next_in = ctypes.addressof(src)
        self.s.avail_in = len(data)
        obuf = ctypes.create_string_buffer(out_chunk)
        while True:
            self.s.next_out = ctypes.addressof(obuf)
            self.s.avail_out = out_chunk
            rc = L().inflate(ctypes.byref(self.s), flush)
            self.out += obuf.raw[: out_chunk - self.s.avail_out]
            if rc != Z_OK or self.s.avail_out != 0:
                return rc

    def end(self):
        return L().inflateEnd(ctypes.byref(self.s))


@pytest.mark.parametrize("chunk", [1 << 16, 16384, 4099, 257])
def test_streaming_inflate_large_stream_in_chunks(chunk):
    """zpipe's loop on a stream of several MiB: output arrives as the blocks complete, Z_STREAM_END on the call that brings the
    last byte, nothing quadratic (advisor: inputs over 1 MiB never finished)."""
    d = silesia_tar()[: 6 << 20] if chunk >= 4099 else silesia_member(3)[:300000]  # text: several blocks even in 300 KB
    comp = zlib.compress(d, 6)
    z = Inf()
    rc = Z_OK
    first_out_at = None
    for i in range(0, len(comp), chunk):
        assert rc in (Z_OK, Z_BUF_ERROR)
        rc = z.feed(comp[i:i + chunk])
        if z.out and first_out_at is None:
            first_out_at = i
    assert rc == Z_STREAM_END and bytes(z.out) == d
    assert z.s.total_in == len(comp) and z.s.total_out == len(d) and z.s.adler == zlib.adler32(d)
    assert first_out_at is not None and first_out_at < len(comp) // 2, "output must not wait for the end of the stream"
    assert z.end() == Z_OK


def test_streaming_inflate_bytes_behind_the_stream_stay_with_the_caller():
    d = synthetic_mix(50000, seed=3)
    comp = zlib.compress(d, 6)
    z = Inf()
    rc = z.feed(comp + b"TRAILING!")
    assert rc == Z_STREAM_END and bytes(z.out) == d and z.s.avail_in == 9 and z.s.total_in == len(comp)
    # concatenated members: reset and go on with what was left
    two = comp + zlib.compress(d[::-1], 9)
    z2 = Inf()
    assert z2.feed(two) == Z_STREAM_END
    left = z2.s.avail_in
    assert left == len(two) - len(comp)
    assert L().inflateReset(ctypes.byref(z2.s)) == Z_OK
    z2.out = bytearray()
    assert z2.feed(two[len(comp):]) == Z_STREAM_END and bytes(z2.out) == d[::-1]


def test_input_ending_on_block_boundaries_is_not_a_data_error():
    """Advisor: a prefix that ends exactly behind a sync marker, behind a stored block or inside LEN/NLEN is 'need more input'."""
    d = synthetic_mix(120000, seed=5)
    co = zlib.compressobj(6)
    parts = [co.compress(d[:40000]) + co.flush(zlib.Z_SYNC_FLUSH), co.compress(d[40000:80000]) + co.flush(zlib.Z_FULL_FLUSH),
             co.compress(d[80000:]) + co.flush()]
    comp = b"".join(parts)
    cuts = [len(parts[0]), len(parts[0]) - 2, len(parts[0]) - 4, len(parts[0]) + len(parts[1]), len(parts[0]) + len(parts[1]) - 1]
    st = zlib.compressobj(0)
    stored = st.compress(d[:70000]) + st.flush()
    for stream, cutlist in ((comp, cuts), (stored, [2 + 5 + 65535, 2 + 3, 2 + 5 + 65535 + 2, 2 + 1])):
        for cut in cutlist:
            z = Inf()
            rc = z.feed(stream[:cut])
            assert rc in (Z_OK, Z_BUF_ERROR), (cut, rc, z.s.msg)
            rc = z.feed(stream[cut:])
            assert rc == Z_STREAM_END and bytes(z.out) == zlib.decompress(stream), cut
    # the sync point of the reference: stopped in front of LEN/NLEN of the empty stored block
    z = Inf()
    z.feed(parts[0][:-4])
    assert L().inflateSyncPoint(ctypes.byref(z.s)) == 1
    z.feed(parts[0][-4:])
    assert L().inflateSyncPoint(ctypes.byref(z.s)) == 0
    # the library's own Z_SYNC_FLUSH output, fed as it is produced
    zd = Z.Deflate(6)
    a = zd.deflate(d[:60000], Z.Z_SYNC_FLUSH)
    zi = Inf()
    assert zi.feed(a) in (Z_OK, Z_BUF_ERROR) and bytes(zi.out) == d[:60000]
    b = zd.deflate(d[60000:], Z.Z_FINISH)
    assert zi.feed(b) == Z_STREAM_END and bytes(zi.out) == d


def test_truncated_streams_whose_zero_code_is_a_literal_terminate():
    """Advisor: the block scan must not run forever on the zero padding behind a truncated input."""
    found = 0
    for k in (2, 5, 1, 9):
        d = silesia_member(k)[:900000]
        comp = zlib.compress(d, 6)
        for cut in range(70000, len(comp) - 8, 16384):
            with pytest.raises(Z.ZlibError) as ei:
                Z.uncompress(comp[:cut], len(d))
            assert ei.value.code in (Z_DATA_ERROR, Z_BUF_ERROR)
            found += 1
            if found > 40:
                return


def test_gzip_header_fields_both_ways():
    """deflateSetHeader emits the fields (the reference's gzip_with_header check: 81 bytes, zlib-rs/src/deflate.rs:3897-3985) and
    inflateGetHeader returns them; FHCRC is verified."""
    lib = L()
    # the reference's own case first: "Hello World\n", extra / name / comment / hcrc -> 81 bytes
    ref = O.gzip_with_header(b"Hello World\n", 6, extra=b"some extra stuff\0", name=b"nomen est omen\0", comment=b"such comment\0", hcrc=1)
    assert len(ref) == 81
    extra, name, comment = b"some extra stuff\0", b"nomen est omen\0", b"such comment\0"
    for data, kw in ((b"Hello World\n", dict(text=0, time=0, os=0)),):
        eb, nb, cb = (ctypes.create_string_buffer(x, len(x)) for x in (extra, name, comment))
        h = GzHeader(text=0, time=0, xflags=0, os=0, extra=ctypes.addressof(eb), extra_len=len(extra), extra_max=0,
                     name=ctypes.addressof(nb), name_max=0, comment=ctypes.addressof(cb), comm_max=0, hcrc=1, done=0)
        s = Z.ZStream()
        assert lib.deflateInit2_(ctypes.byref(s), 6, 8, 31, 8, 0, Z.ZLIB_VERSION, ctypes.sizeof(Z.ZStream)) == Z_OK
        assert lib.deflateSetHeader(ctypes.byref(s), ctypes.byref(h)) == Z_OK
        src = ctypes.create_string_buffer(data, len(data))
        dst = ctypes.create_string_buffer(512)
        s.next_in, s.avail_in, s.next_out, s.avail_out = ctypes.addressof(src), len(data), ctypes.addressof(dst), 512
        assert lib.deflate(ctypes.byref(s), Z_FINISH) == Z_STREAM_END
        assert dst.raw[: s.total_out] == ref
        lib.deflateEnd(ctypes.byref(s))
    extra, name, comment = b"\x01\x02\x03\x04\x05", b"test.txt\0", b"a gzip comment\0"
    eb, nb, cb = (ctypes.create_string_buffer(x, len(x)) for x in (extra, name, comment))
    h = GzHeader(text=1, time=1234567, xflags=0, os=3, extra=ctypes.addressof(eb), extra_len=len(extra), extra_max=0,
                 name=ctypes.addressof(nb), name_max=0, comment=ctypes.addressof(cb), comm_max=0, hcrc=1, done=0)
    data = b"Hello World!\n" * 3
    s = Z.ZStream()
    assert lib.deflateInit2_(ctypes.byref(s), 6, 8, 31, 8, 0, Z.ZLIB_VERSION, ctypes.sizeof(Z.ZStream)) == Z_OK
    assert lib.deflateSetHeader(ctypes.byref(s), ctypes.byref(h)) == Z_OK
    src = ctypes.create_string_buffer(data, len(data))
    dst = ctypes.create_string_buffer(512)
    s.next_in, s.avail_in, s.next_out, s.avail_out = ctypes.addressof(src), len(data), ctypes.addressof(dst), 512
    assert lib.deflate(ctypes.byref(s), Z_FINISH) == Z_STREAM_END
    out = dst.raw[: s.total_out]
    used = ctypes.c_int(0)
    assert lib.deflateUsed(ctypes.byref(s), ctypes.byref(used)) == Z_OK and 1 <= used.value <= 8
    assert lib.deflateEnd(ctypes.byref(s)) == Z_OK
    want = O.gzip_with_header(data, 6, text=1, time=1234567, os=3, extra=extra, name=name, comment=comment, hcrc=1)
    assert out == want
    import gzip
    assert gzip.decompress(out) == data
    # read it back
    z = Inf(31)
    g = GzHeader()
    xb, nb2, cb2 = ctypes.create_string_buffer(64), ctypes.create_string_buffer(64), ctypes.create_string_buffer(64)
    g.extra, g.extra_max, g.name, g.name_max, g.comment, g.comm_max = ctypes.addressof(xb), 64, ctypes.addressof(nb2), 64, ctypes.addressof(cb2), 64
    assert lib.inflateGetHeader(ctypes.byref(z.s), ctypes.byref(g)) == Z_OK
    assert z.feed(out) == Z_STREAM_END and bytes(z.out) == data
    assert g.done == 1 and g.text == 1 and g.time == 1234567 and g.os == 3 and g.hcrc == 1
    assert xb.raw[: g.extra_len] == extra and nb2.value + b"\0" == name and cb2.value + b"\0" == comment
    # a damaged header crc is rejected with the reference's message
    bad = bytearray(out)
    hdr_len = 10 + 2 + len(extra) + len(name) + len(comment)
    bad[hdr_len] ^= 0x55
    zb = Inf(31)
    assert zb.feed(bytes(bad)) == Z_DATA_ERROR and zb.s.msg == b"header crc mismatch"
    # zlib-wrapped streams take no gzip header
    s2 = Z.ZStream()
    assert lib.deflateInit_(ctypes.byref(s2), 6, Z.ZLIB_VERSION, ctypes.sizeof(Z.ZStream)) == Z_OK
    assert lib.deflateSetHeader(ctypes.byref(s2), ctypes.byref(h)) == Z_STREAM_ERROR
    assert lib.deflateTune(ctypes.byref(s2), 8, 16, 128, 128) == Z_OK      # the level's own parameters
    assert lib.deflateTune(ctypes.byref(s2), 4, 4, 8, 4) == Z_STREAM_ERROR   # anything else is refused, not ignored
    lib.deflateEnd(ctypes.byref(s2))


def test_inflate_with_preset_dictionary_and_get_dictionary():
    lib = L()
    d = synthetic_mix(90000, seed=9)
    zdict = d[20000:50000]
    co = zlib.compressobj(6, zlib.DEFLATED, 15, 8, zlib.Z_DEFAULT_STRATEGY, zdict)
    comp = co.compress(d) + co.flush()
    z = Inf()
    assert z.feed(comp) == Z_NEED_DICT and z.s.adler == zlib.adler32(zdict)
    wrong = ctypes.create_string_buffer(b"not the dictionary", 18)
    assert lib.inflateSetDictionary(ctypes.byref(z.s), ctypes.addressof(wrong), 18) == Z_DATA_ERROR
    db = ctypes.create_string_buffer(zdict, len(zdict))
    assert lib.inflateSetDictionary(ctypes.byref(z.s), ctypes.addressof(db), len(zdict)) == Z_OK
    assert z.feed(b"") == Z_STREAM_END and bytes(z.out) == d and z.s.adler == zlib.adler32(d)
    win = ctypes.create_string_buffer(32768)
    n = ctypes.c_uint(0)
    assert lib.inflateGetDictionary(ctypes.byref(z.s), ctypes.addressof(win), ctypes.byref(n)) == Z_OK
    assert n.value == 32768 and win.raw == d[-32768:]
    # raw stream: the dictionary may be set up front
    cr = zlib.compressobj(6, zlib.DEFLATED, -15, 8, zlib.Z_DEFAULT_STRATEGY, zdict)
    raw = cr.compress(d) + cr.flush()
    zr = Inf(-15)
    assert lib.inflateSetDictionary(ctypes.byref(zr.s), ctypes.addressof(db), len(zdict)) == Z_OK
    assert zr.feed(raw[:1000]) in (Z_OK, Z_BUF_ERROR)
    assert zr.feed(raw[1000:]) == Z_STREAM_END and bytes(zr.out) == d
    # a zlib stream without FDICT refuses a dictionary (inflate.rs:2622)
    zz = Inf()
    assert lib.inflateSetDictionary(ctypes.byref(zz.s), ctypes.addressof(db), len(zdict)) == Z_STREAM_ERROR


def test_inflate_sync_skips_to_the_next_flush_marker():
    lib = L()
    d = synthetic_mix(100000, seed=11)
    co = zlib.compressobj(6)
    a = co.compress(d[:50000]) + co.flush(zlib.Z_FULL_FLUSH)
    b = co.compress(d[50000:]) + co.flush()
    damaged = bytearray(a + b)
    damaged[len(a) // 2] ^= 0xff
    z = Inf()
    rc = z.feed(bytes(damaged[: len(a)]))
    if rc not in (Z_DATA_ERROR,):  # the damage may only show in the check value; force the sync either way
        pass
    tail = bytes(damaged[len(a) - 6:])  # the marker 00 00 ff ff is in the last four bytes of `a`
    src = ctypes.create_string_buffer(tail, len(tail))
    z.s.next_in, z.s.avail_in = ctypes.addressof(src), len(tail)
    assert lib.inflateSync(ctypes.byref(z.s)) == Z_OK
    z.out = bytearray()
    rest = tail[len(tail) - z.s.avail_in:]
    rc = z.feed(rest)
    assert rc in (Z_STREAM_END, Z_OK, Z_BUF_ERROR) and bytes(z.out) == d[50000:]
    # no marker: Z_DATA_ERROR
    z2 = Inf()
    junk = ctypes.create_string_buffer(b"\x01\x02\x03\x04\x05\x06\x07", 7)
    z2.s.next_in, z2.s.avail_in = ctypes.addressof(junk), 7
    assert lib.inflateSync(ctypes.byref(z2.s)) == Z_DATA_ERROR


def test_inflate_back_and_misc_exports():
    lib = L()
    zs = ctypes.POINTER(Z.ZStream)
    IN = ctypes.CFUNCTYPE(ctypes.c_uint, ctypes.c_void_p, ctypes.POINTER(ctypes.c_void_p))
    OUT = ctypes.CFUNCTYPE(ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_uint)
    lib.inflateBackInit_.argtypes = [zs, ctypes.c_int, ctypes.c_void_p, ctypes.c_char_p, ctypes.c_int]
    lib.inflateBack.argtypes = [zs, IN, ctypes.c_void_p, OUT, ctypes.c_void_p]
    lib.inflateBackEnd.argtypes = [zs]
    d = synthetic_mix(200000, seed=13)
    cr = zlib.compressobj(6, zlib.DEFLATED, -15)
    raw = cr.compress(d) + cr.flush()
    chunks = [raw[i:i + 9000] for i in range(0, len(raw), 9000)]
    keep, got, state = [], bytearray(), {"i": 0}

    def fin(_, pp):
        if state["i"] >= len(chunks):
            return 0
        b = ctypes.create_string_buffer(chunks[state["i"]], len(chunks[state["i"]]))
        keep.append(b)
        state["i"] += 1
        pp[0] = ctypes.addressof(b)
        return len(b)

    def fout(_, p, n):
        got.extend(ctypes.string_at(p, n))
        return 0

    s = Z.ZStream()
    win = ctypes.create_string_buffer(32768)
    assert lib.inflateBackInit_(ctypes.byref(s), 15, ctypes.addressof(win), Z.ZLIB_VERSION, ctypes.sizeof(Z.ZStream)) == Z_OK
    assert lib.inflateBack(ctypes.byref(s), IN(fin), None, OUT(fout), None) == Z_STREAM_END
    assert bytes(got) == d
    assert lib.inflateBackEnd(ctypes.byref(s)) == Z_OK
    assert lib.inflateBackInit_(ctypes.byref(s), 15, None, Z.ZLIB_VERSION, ctypes.sizeof(Z.ZStream)) == Z_STREAM_ERROR
    # get_crc_table is the byte-wise table of the reflected polynomial
    lib.get_crc_table.restype = ctypes.POINTER(ctypes.c_uint32 * 256)
    t = lib.get_crc_table().contents
    assert t[0] == 0 and t[1] == 0x77073096 and t[255] == 0x2d02ef8d
    z = Inf()
    assert lib.inflateMark(ctypes.byref(z.s)) == -65536
    assert lib.inflateValidate(ctypes.byref(z.s), 0) == Z_OK
    comp = bytearray(zlib.compress(d[:5000], 6))
    comp[-1] ^= 1  # a wrong adler32 is not looked at any more
    assert z.feed(bytes(comp)) == Z_STREAM_END and bytes(z.out) == d[:5000]
    # inflatePrime: resume a raw stream behind a block that ended inside a byte
    co = zlib.compressobj(6, zlib.DEFLATED, -15)
    first = co.compress(d[:30000]) + co.flush(zlib.Z_SYNC_FLUSH)
    second = co.compress(d[30000:60000]) + co.flush()
    zp = Inf(-15)
    assert zp.feed(first) in (Z_OK, Z_BUF_ERROR) and bytes(zp.out) == d[:30000]
    zp2 = Inf(-15)
    db = ctypes.create_string_buffer(d[:30000][-32768:], min(30000, 32768))
    assert lib.inflateSetDictionary(ctypes.byref(zp2.s), ctypes.addressof(db), len(db)) == Z_OK
    assert lib.inflatePrime(ctypes.byref(zp2.s), 3, second[0] & 7) == Z_OK
    shifted = bytes(((second[i] >> 3) | ((second[i + 1] << 5) & 0xff)) if i + 1 < len(second) else (second[i] >> 3) for i in range(len(second)))
    assert zp2.feed(shifted) in (Z_STREAM_END, Z_OK, Z_BUF_ERROR) and bytes(zp2.out) == d[30000:60000]


def deflate_with_dict(data, zdict, level=6, wbits=15, strategy=0, mem_level=8):
    """deflateInit2 + deflateSetDictionary + deflate(Z_FINISH) through the ABI.  Returns (stream, dictid as left in strm.adler)."""
    lib = L()
    lib.deflateSetDictionary.argtypes = [ctypes.POINTER(Z.ZStream), ctypes.c_void_p, ctypes.c_uint]
    s = Z.ZStream()
    assert lib.deflateInit2_(ctypes.byref(s), level, 8, wbits, mem_level, strategy, Z.ZLIB_VERSION, ctypes.sizeof(Z.ZStream)) == Z_OK
    db = ctypes.create_string_buffer(bytes(zdict), max(len(zdict), 1))
    assert lib.deflateSetDictionary(ctypes.byref(s), ctypes.addressof(db), len(zdict)) == Z_OK
    did = s.adler
    src = ctypes.create_string_buffer(bytes(data), max(len(data), 1))
    cap = len(data) + len(data) // 8 + 1024
    dst = ctypes.create_string_buffer(cap)
    s.next_in, s.avail_in, s.next_out, s.avail_out = ctypes.addressof(src), len(data), ctypes.addressof(dst), cap
    assert lib.deflate(ctypes.byref(s), Z_FINISH) == Z_STREAM_END
    out = dst.raw[: s.total_out]
    assert lib.deflateEnd(ctypes.byref(s)) == Z_OK
    return out, did


@pytest.mark.parametrize("level", [0, 3, 4, 5, 6, 7, 8, 9])
def test_deflate_with_preset_dictionary_bit_exact(level):
    """deflate::set_dictionary (zlib-rs/src/deflate.rs:498-564): the stream (FDICT header, dictionary id, data parsed against the
    dictionary, adler32 of the input) equals the oracle's for every dictionary length class (short, one window, more than one
    window, more than the window buffer) and for inputs on the serial and on the parallel path."""
    m = silesia_member(3)
    x = silesia_member(9)
    for dl, n in ((5, 14), (1000, 3000), (32768, 200000), (40000, 120000), (70000, 300000), (2, 5000), (3, 70000)):
        for src in (m, x):
            dic, data = src[:dl], src[dl: dl + n]
            rc, want, did = O.compress_dict(data, dic, level)
            assert rc == 0
            got, gid = deflate_with_dict(data, dic, level)
            assert gid == did == zlib.adler32(dic)
            assert got == want, (level, dl, n, len(got), len(want))
            assert zlib.decompressobj(zdict=dic).decompress(got) == data


def test_deflate_dictionary_reference_case_strategies_and_ghost_entry():
    # the reference's own check (test-libz-rs-sys/src/deflate.rs:862-900): "hello" / "hello, hello!\0"
    rc, want, did = O.compress_dict(b"hello, hello!\0", b"hello", 6)
    got, gid = deflate_with_dict(b"hello, hello!\0", b"hello", 6)
    assert got == want and gid == did
    d = synthetic_mix(150000, seed=21)
    for strategy in (1, 2, 3, 4):
        for level in (6, 9):
            rc, want, did = O.compress_dict(d[3000:], d[:3000], level, 15, 8, strategy)
            got, _ = deflate_with_dict(d[3000:], d[:3000], level, 15, strategy)
            assert got == want, (strategy, level)
    # raw stream: no header, no check value
    rc, want, did = O.compress_dict(d[1000:90000], d[:1000], 6, -15)
    got, _ = deflate_with_dict(d[1000:90000], d[:1000], 6, -15)
    assert got == want
    # the last dictionary string is first hashed with a zero behind it (deflate.rs:535-545): an input that continues with a
    # non-zero byte and soon repeats "<last three dictionary bytes> 0" walks through that stale table entry
    dic = bytes(range(50, 250)) * 4 + b"abc"
    for filler in (40, 300, 5000):
        data = b"Xyz" + bytes((i * 7 + 3) % 251 + 1 for i in range(filler)) + b"abc\0abc\0abcX" + d[:60000]
        for level in (4, 6, 8):
            rc, want, did = O.compress_dict(data, dic, level)
            got, _ = deflate_with_dict(data, dic, level)
            assert got == want, (filler, level)
    # gzip streams take no dictionary; a zlib stream only before the first deflate() call
    lib = L()
    s = Z.ZStream()
    assert lib.deflateInit2_(ctypes.byref(s), 6, 8, 31, 8, 0, Z.ZLIB_VERSION, ctypes.sizeof(Z.ZStream)) == Z_OK
    db = ctypes.create_string_buffer(b"dict", 4)
    assert lib.deflateSetDictionary(ctypes.byref(s), ctypes.addressof(db), 4) == Z_STREAM_ERROR
    lib.deflateEnd(ctypes.byref(s))


def test_mixed_flush_sequence_and_deflate_prime():
    """Segments that end inside a byte (Z_PARTIAL_FLUSH, Z_BLOCK) hand their last bits to the next segment; the previous input is the
    next segment's window (not after Z_FULL_FLUSH).  The stitched stream is what stock zlib inflates; deflatePrime puts bits in front
    of a raw stream (zlib-rs/src/deflate.rs:566-604)."""
    d = silesia_member(3)[:400000]
    flushes = [Z.Z_PARTIAL_FLUSH, Z.Z_BLOCK, Z.Z_SYNC_FLUSH, Z.Z_BLOCK, Z.Z_PARTIAL_FLUSH, Z.Z_FULL_FLUSH, Z.Z_BLOCK, Z.Z_NO_FLUSH]
    for wbits in (15, -15, 31):
        z = Z.Deflate(6, window_bits=wbits)
        out = bytearray()
        step = len(d) // len(flushes)
        for i, f in enumerate(flushes):
            out += z.deflate(d[i * step:(i + 1) * step], f)
        out += z.deflate(d[len(flushes) * step:], Z.Z_FINISH)
        assert zlib.decompress(bytes(out), wbits) == d
        if wbits == 15:
            one = zlib.compress(d, 6)
            assert len(out) < len(one) * 1.02  # the window survives the flushes: hardly any ratio is lost
    # deflatePrime: 5 bits in front of a raw stream; dropping them again gives a stream that inflates
    lib = L()
    lib.deflatePrime.argtypes = [ctypes.POINTER(Z.ZStream), ctypes.c_int, ctypes.c_int]
    s = Z.ZStream()
    assert lib.deflateInit2_(ctypes.byref(s), 6, 8, -15, 8, 0, Z.ZLIB_VERSION, ctypes.sizeof(Z.ZStream)) == Z_OK
    assert lib.deflatePrime(ctypes.byref(s), 5, 0b10110) == Z_OK
    data = d[:50000]
    src = ctypes.create_string_buffer(data, len(data))
    dst = ctypes.create_string_buffer(len(data))
    s.next_in, s.avail_in, s.next_out, s.avail_out = ctypes.addressof(src), len(data), ctypes.addressof(dst), len(data)
    assert lib.deflate(ctypes.byref(s), Z_FINISH) == Z_STREAM_END
    out = dst.raw[: s.total_out]
    lib.deflateEnd(ctypes.byref(s))
    assert out[0] & 31 == 0b10110
    bits = int.from_bytes(out, "little") >> 5
    assert zlib.decompress(bits.to_bytes(len(out), "little"), -15) == data


def test_reference_zpipe_binary_round_trip(tmp_path):
    """The reference's zpipe.c, built unchanged against this library by build() (oracle/_ref/zpipe_ref), compresses and
    decompresses a file of several MiB through 16 KiB deflate()/inflate() calls."""
    import subprocess
    exe = os.path.join(os.path.dirname(HERE), "oracle", "_ref", "zpipe_ref")
    if not os.path.exists(exe):
        pytest.skip("oracle/_ref/zpipe_ref was not built (no zlib-rs source tree at build time)")
    d = silesia_tar()[: 5 << 20]
    env = dict(os.environ, LD_LIBRARY_PATH=os.path.join(os.path.dirname(HERE), "zlib_rs_b200"))
    z = subprocess.run([exe], input=d, capture_output=True, timeout=600, env=env)
    assert z.returncode == 0, z.stderr[-500:]
    assert zlib.decompress(z.stdout) == d and z.stdout == O.compress(d, 6)[1]  # Z_DEFAULT_COMPRESSION through deflate(Z_FINISH) at EOF
    u = subprocess.run([exe, "-d"], input=z.stdout, capture_output=True, timeout=600, env=env)
    assert u.returncode == 0 and u.stdout == d
