"""GPU (B200): the CUDA path, called through the C ABI, against the oracle side.

Bars (BASELINE.json north_star): valid brotli stream; bit-exact round trip through an independent decoder;
compressed size <= +0.5 % of the reference restatement at the same quality / lgwin; and -- stronger than required --
bit identity with the CPU model of the pipeline (integer work: every stage is deterministic)."""
import hashlib
import io

import numpy as np
import pytest

from conftest import assert_size_parity, golden_bytes
from oracle.harness import sys_compress, sys_decompress

pytestmark = pytest.mark.gpu

FILES = ["alice29.txt", "asyoulik.txt", "random_then_unicode", "quickfox_repeated", "random_org_10k.bin", "backward65536",
         "64x", "ukkonooa", "monkey", "x", "xyzzy", "10x10y", "aaabaaaa", "empty", "quickfox", "compressed_file"]


@pytest.mark.parametrize("name", FILES)
@pytest.mark.parametrize("q,w", [(5, 20), (5, 22), (7, 22), (9, 22), (9, 16), (5, 18), (10, 22), (11, 22), (11, 24), (10, 16)])
def test_fixture_parity(encoder, golden_table, name, q, w):
    d = golden_bytes(name)
    c = encoder.compress(d, q, w)
    assert sys_decompress(c, max(len(d), 1)) == d
    g = golden_table["%s|q%d|w%d" % (name, q, w)]
    assert hashlib.sha256(c).hexdigest() == g["model_sha256"], "GPU stream differs from the CPU model"
    # reference size = the restatement without static dictionary, or Google's encoder with it, whichever is larger (on
    # tiny inputs dictionary references cost a few bytes: quickfox_repeated is 46 B without, 51 B with)
    assert len(c) <= max(g["oracle_size"], g["libbrotlienc_size"]) * 1.005 + 8


def test_config1_alice29_q5_w20(encoder, oracle):
    """BASELINE config 1: alice29.txt, quality 5, lgwin 20."""
    d = golden_bytes("alice29.txt")
    c = encoder.compress(d, 5, 20)
    assert sys_decompress(c, len(d)) == d
    ref, _ = oracle.compress(d, 5, 20)
    assert len(c) <= len(ref) * 1.005
    # vs Google's C encoder (the code the reference is a port of; it also matches static-dictionary words): within 0.5 %
    assert len(c) <= len(sys_compress(d, 5, 20)) * 1.005


def test_product_against_reference_held_pins(encoder):
    """The reference's own size vectors for this quality range, asserted on the PRODUCT (not on the oracle):
    alice29.txt q9 lgwin16 one-shot = 51 737 B exactly (src/enc/encode.rs:3073-3091); alice29.txt lgwin 22 quality 10 = 47 488 B
    and quality 11 = 46 493 B (src/bin/integration_tests.rs:408-449) -> each within +-0.5 %."""
    d = golden_bytes("alice29.txt")
    for q, w, pin in ((9, 16, 51737), (10, 22, 47488), (11, 22, 46493)):
        c = encoder.compress(d, q, w)
        assert sys_decompress(c, len(d)) == d
        assert abs(len(c) - pin) <= pin * 0.005, (q, w, len(c), pin)


def test_custom_dictionary_and_abi_details():
    """BrotliEncoderSetCustomDictionary (src/ffi/compressor.rs:162): the dictionary becomes window content in front of the
    stream -- the stream only decodes with the same dictionary attached; total_out is the cumulative count."""
    import ctypes
    import rust_brotli_b200 as rb
    L = rb._capi()
    d = golden_bytes("alice29.txt")
    dictionary, payload = d[:60000], d[50000:120000]
    outs = []
    for use_dict in (False, True):
        h = L.BrotliEncoderCreateInstance(None, None, None)
        assert h
        assert L.BrotliEncoderSetParameter(h, rb.BROTLI_PARAM_QUALITY, 5)
        assert not L.BrotliEncoderSetParameter(h, rb.BROTLI_PARAM_LARGE_WINDOW, 1)
        if use_dict:
            L.BrotliEncoderSetCustomDictionary(h, len(dictionary), dictionary)
        buf = ctypes.create_string_buffer(len(payload) + 4096)
        avail_in, avail_out = ctypes.c_size_t(len(payload)), ctypes.c_size_t(len(buf))
        next_in = ctypes.c_void_p(ctypes.cast(ctypes.c_char_p(payload), ctypes.c_void_p).value)
        next_out = ctypes.c_void_p(ctypes.addressof(buf))
        total = ctypes.c_size_t(12345)  # garbage in: the call assigns the cumulative total (encode.rs:1591-1593)
        assert L.BrotliEncoderCompressStream(h, rb.BROTLI_OPERATION_FINISH, ctypes.byref(avail_in), ctypes.byref(next_in),
                                             ctypes.byref(avail_out), ctypes.byref(next_out), ctypes.byref(total))
        n = len(buf) - avail_out.value
        assert total.value == n and L.BrotliEncoderIsFinished(h)
        outs.append(buf.raw[:n])
        L.BrotliEncoderDestroyInstance(h)
    plain, with_dict = outs
    assert sys_decompress(plain, len(payload)) == payload
    from oracle.harness import sys_decompress_with_dictionary
    assert sys_decompress_with_dictionary(with_dict, len(payload), dictionary) == payload
    assert len(with_dict) < 0.9 * len(plain)  # the first 10 000 bytes of the payload are literally in the dictionary


def test_match_stage_equals_model(encoder, model):
    """Per-position best bucket match (distance << 8 | capped length): CUDA sort+match vs the sequential ring model."""
    d = (golden_bytes("random_then_unicode") + golden_bytes("alice29.txt"))[:400000]
    for q, w in ((5, 22), (9, 18)):
        got = encoder.stage_match(d, q, w)
        ref = np.zeros(len(d), dtype=np.uint32)
        model.compress(d, q, w, best_out=ref.ctypes.data)
        assert np.array_equal(got, ref)


@pytest.mark.parametrize("n", [0, 1, 2, 3, 7, 8, 9, 63, 64, 65, 4095, 4096, 4097, 8191, 8192, 12289, 65536, 65537])
def test_edge_sizes(encoder, model, n):
    d = (golden_bytes("alice29.txt") * 2)[:n]
    c = encoder.compress(d, 5, 22)
    assert sys_decompress(c, max(n, 1)) == d
    assert c == model.compress(d, 5, 22)[0]


@pytest.mark.parametrize("q", [9, 10, 11])
def test_edge_sizes_deep_and_hq(encoder, model, q):
    """The sizes that switch something on in the q9 on-demand search (forced) and in the q10 / q11 path: first bucket match, the
    long-prefix levels (8 + 8 / 16 / 32 bytes), the 512-byte warm-up, 8 / 16 KiB parse units, the 64 KiB statistics window."""
    import rust_brotli_b200 as rb
    src = golden_bytes("alice29.txt") * 2
    encoder.set_option(rb._native.OPT_ONDEMAND, 2)
    try:
        for n in (0, 1, 2, 3, 7, 8, 9, 39, 40, 41, 63, 64, 65, 511, 512, 513, 4097, 8191, 8192, 8193, 16383, 16385, 65535, 65537, 70001):
            d = src[:n]
            c = encoder.compress(d, q, 22)
            assert sys_decompress(c, max(n, 1)) == d, n
            assert c == model.compress(d, q, 22)[0], n
    finally:
        encoder.set_option(rb._native.OPT_ONDEMAND, 1)


@pytest.mark.parametrize("lgwin", [10, 12, 16, 17, 18, 20, 24])
def test_window_sizes(encoder, model, lgwin):
    d = golden_bytes("asyoulik.txt") + golden_bytes("alice29.txt")
    c = encoder.compress(d, 6, lgwin)
    assert sys_decompress(c, len(d)) == d
    assert c == model.compress(d, 6, lgwin)[0]


def test_incompressible_and_degenerate(encoder, model):
    from tools import datagen
    for d in (datagen.pcg_random(1_500_000), bytes(3_000_000), datagen.tiled(golden_bytes("random_org_10k.bin"), 5_000_000),
              datagen.tiled(golden_bytes("quickfox_repeated"), 6_000_000)):
        c = encoder.compress(d, 5, 22)
        assert sys_decompress(c, len(d)) == d
        assert c == model.compress(d, 5, 22)[0]
        assert len(c) <= len(d) + 64


def test_multi_chunk_stream_equals_model(encoder, model):
    """Streams longer than one 24 MiB chunk: chunks run on alternating lanes (streams) and append to one bit stream; the
    result must not depend on the number of lanes and must equal the model's chunk loop."""
    import rust_brotli_b200 as rb
    from tools import datagen
    d = datagen.enwik_like(30_000_000) + datagen.pcg_random(22_000_000)[:21_000_000] + golden_bytes("alice29.txt") * 20
    ref = model.compress(d, 5, 22)[0]
    for lanes in (2, 1, 2):
        encoder.set_option(rb._native.OPT_LANES, lanes)
        c = encoder.compress(d, 5, 22)
        assert c == ref, "lanes=%d" % lanes
    assert sys_decompress(ref, len(d)) == d


def test_long_stream_is_emitted_in_pieces():
    """CompressorWriter fed 230 MB in 8 MiB writes: PROCESS emits byte-aligned 96 MiB pieces while input keeps arriving and
    keeps only the match window of what is already emitted (bounded host buffer); the concatenation is one valid stream."""
    import rust_brotli_b200 as rb
    from tools import datagen
    base = datagen.enwik_like(23_000_000, seed=5)
    sink = io.BytesIO()
    w = rb.CompressorWriter(sink, 4096, 5, 22)
    emitted_before_close = 0
    for rep in range(10):
        for o in range(0, len(base), 8 << 20):
            w.write(base[o:o + (8 << 20)])
        emitted_before_close = sink.tell()
    w.close()
    assert emitted_before_close > 0, "no output before FINISH"
    out = sink.getvalue()
    assert sys_decompress(out, 10 * len(base)) == base * 10


def test_large_window_multi_batch(encoder, model):
    """lgwin 24: the window (16 MiB) is most of a 2^25-position sort batch, so a 24 MiB chunk takes two batches and the second
    chunk sees a halo longer than itself; the stream must equal the model's across both kinds of seam."""
    from tools import datagen
    d = datagen.enwik_like(28_000_000, seed=3)
    c = encoder.compress(d, 5, 24)
    assert sys_decompress(c, len(d)) == d
    assert c == model.compress(d, 5, 24)[0]


def test_structured_logs_size_parity(encoder, oracle):
    """Record-structured JSON logs lean on the distance cache: the warm-up in front of every parse unit keeps the size
    within +0.5 % of the reference restatement (it was +1.4 % with units that start from an unknown cache)."""
    from tools import datagen
    d = datagen.json_logs(4_000_000)
    for q in (5, 9):
        c = encoder.compress(d, q, 22)
        assert sys_decompress(c, len(d)) == d
        assert len(c) <= len(oracle.compress(d, q, 22)[0]) * 1.005


def test_static_dictionary_toggle(encoder, model):
    """Static-dictionary references (distances beyond the window) decode, equal the model, and pay off on English text."""
    import rust_brotli_b200 as rb
    d = golden_bytes("asyoulik.txt")
    on = encoder.compress(d, 5, 22)
    encoder.set_option(rb._native.OPT_DICT, 0)
    try:
        off = encoder.compress(d, 5, 22)
    finally:
        encoder.set_option(rb._native.OPT_DICT, 1)
    assert sys_decompress(on, len(d)) == d and sys_decompress(off, len(d)) == d
    assert on == model.compress(d, 5, 22)[0] and off == model.compress(d, 5, 22, use_dict=0)[0]
    assert len(on) < len(off)


def test_long_literal_runs(encoder, model):
    """Inserts longer than LONG_INS literals take the segment kernels (k_symbols_long / k_bitlen_long / k_emit_long):
    text interleaved with incompressible runs of many lengths, including runs that cross literal block switches."""
    from tools import datagen
    text = golden_bytes("alice29.txt")
    rnd = datagen.pcg_random(3_000_000)
    parts, o, t = [], 0, 0
    for run in (511, 512, 513, 600, 1023, 1024, 1025, 5000, 70_000, 1_500_000, 200_000, 513):
        parts.append(text[t:t + 20_000]); t = (t + 20_000) % 100_000
        parts.append(rnd[o:o + run]); o += run
    # low-entropy long runs compress instead of going raw: 3-symbol noise
    parts.append(bytes(b % 3 + 65 for b in rnd[:900_000]))
    parts.append(text)
    d = b"".join(parts)
    for q in (5, 9):
        c = encoder.compress(d, q, 22)
        assert sys_decompress(c, len(d)) == d
        assert c == model.compress(d, q, 22)[0]


def test_multi_metablock_text_size_parity(encoder, model):
    """20 MB of enwik-shaped text (5 metablocks, H6, 13 literal contexts): size within +0.5 % of libbrotlienc q5."""
    from tools import datagen
    d = datagen.enwik_like(20_000_000)
    c = encoder.compress(d, 5, 22)
    assert sys_decompress(c, len(d)) == d
    ref = sys_compress(d, 5, 22)
    assert len(c) <= len(ref) * 1.005, (len(c), len(ref))
    assert c == model.compress(d, 5, 22)[0]


def test_streaming_writer_reader(encoder):
    """src/bin/integration_tests.rs:468-731: CompressorWriter with small writes and a flush per write; CompressorReader."""
    import rust_brotli_b200 as rb
    d = golden_bytes("alice29.txt")
    sink = io.BytesIO()
    w = rb.CompressorWriter(sink, 4096, 5, 22)
    step = 29999
    for i in range(0, len(d), step):
        w.write(d[i:i + step])
        w.flush()
    w.close()
    c = sink.getvalue()
    assert sys_decompress(c, len(d)) == d
    assert len(c) < 0.95 * len(d)
    r = rb.CompressorReader(io.BytesIO(d), 65536, 5, 22)
    c2 = r.read()
    assert sys_decompress(c2, len(d)) == d
    out = io.BytesIO()
    n = rb.BrotliCompress(io.BytesIO(d), out, rb.BrotliEncoderParams(quality=5, lgwin=22))
    assert n == len(out.getvalue()) and sys_decompress(out.getvalue(), len(d)) == d


@pytest.mark.parametrize("threads,q,bound", [(1, 5, 155808), (2, 5, 151857), (3, 5, 144325), (5, 9, 139126)])
def test_compress_multi_bounds(threads, q, bound):
    """src/bin/test_threading.rs:93-124: round trip + size upper bounds on random_then_unicode."""
    import rust_brotli_b200 as rb
    d = golden_bytes("random_then_unicode")
    c = rb.compress_multi(rb.BrotliEncoderParams(quality=q, lgwin=22), d, threads)
    assert sys_decompress(c, len(d)) == d
    assert len(c) <= bound


def test_compress_multi_tiny_inputs():
    """test_threading.rs: empty and 1-byte inputs with 5 threads."""
    import rust_brotli_b200 as rb
    for d in (b"", b"x", b"ab"):
        c = rb.compress_multi(rb.BrotliEncoderParams(quality=5, lgwin=22), d, 5)
        assert sys_decompress(c, max(len(d), 1)) == d


def test_ranges_starting_at_stream_offsets_1_2_3(encoder, model):
    """A range that starts 1 or 2 bytes into the stream has fewer than two context bytes in front of its first literal:
    the missing ones are 0, as the decoder assumes (a guard written as `abs_base || pos >= 2` read data[-1] here)."""
    d = golden_bytes("alice29.txt")[:70000]
    for start in (1, 2, 3):
        head = encoder.compress_range(d, 0, start, 5, 22, True, False, True)
        tail = encoder.compress_range(d, start, len(d) - start, 5, 22, False, True, False)
        assert sys_decompress(head + tail, len(d)) == d
        assert tail == model.compress_range(d, start, len(d) - start, 5, 22, False, True, False)[0]


def test_device_resident_io(encoder):
    """Device pointers in, device pointers out (the `value` path of bench.py)."""
    import torch
    d = golden_bytes("alice29.txt")
    t_in = torch.frombuffer(bytearray(d), dtype=torch.uint8).cuda()
    t_out = torch.empty(len(d) + 65536, dtype=torch.uint8, device="cuda")
    torch.cuda.synchronize()
    n = encoder.compress_device(t_in.data_ptr(), len(d), t_out.data_ptr(), t_out.numel(), 5, 22)
    c = bytes(t_out[:n].cpu().numpy())
    assert sys_decompress(c, len(d)) == d
    assert c == encoder.compress(d, 5, 22)


@pytest.mark.parametrize("q,lgwin", [(9, 22), (8, 22), (7, 22), (9, 16), (5, 16)])
def test_deep_buckets_on_demand_equals_up_front_and_model(encoder, model, q, lgwin):
    """q7..q9 (and lgwin <= 16): the deep bucket lists are searched either for every position up front (k_match_deep + k_parse)
    or on demand where the greedy / lazy walk stands (k_rank_sig + k_parse_ondemand, the reference's own shape:
    FindLongestMatch at the visited positions, backward_references/mod.rs:2376-2552).  Both must give the stream of the CPU
    model, bit for bit -- text, JSON logs and a tail shorter than a unit."""
    import rust_brotli_b200 as rb
    from tools import datagen
    d = datagen.enwik_like(3_000_000) + datagen.json_logs(2_500_000) + golden_bytes("random_then_unicode")[:70001]
    outs = []
    try:
        for mode in (0, 2):
            encoder.set_option(rb._native.OPT_ONDEMAND, mode)
            outs.append(encoder.compress(d, q, lgwin))
    finally:
        encoder.set_option(rb._native.OPT_ONDEMAND, 1)
    assert outs[0] == outs[1]
    assert outs[0] == model.compress(d, q, lgwin)[0]
    assert sys_decompress(outs[0], len(d)) == d
    small = golden_bytes("alice29.txt")  # default rule: a few units stay on the up-front path; forced on demand must agree too
    encoder.set_option(rb._native.OPT_ONDEMAND, 2)
    try:
        forced = encoder.compress(small, q, lgwin)
    finally:
        encoder.set_option(rb._native.OPT_ONDEMAND, 1)
    assert forced == encoder.compress(small, q, lgwin) == model.compress(small, q, lgwin)[0]


# ---- stream framing parameters (SURVEY 8f-2): catable / appendable / magic_number / byte_align / bare_stream ----

def _framed(data, q=5, lgwin=22, **kw):
    import rust_brotli_b200 as rb
    w = io.BytesIO()
    rb.BrotliCompress(io.BytesIO(data), w, rb.BrotliEncoderParams(quality=q, lgwin=lgwin, **kw))
    return w.getvalue()


@pytest.mark.parametrize("q", [5, 9, 10])
def test_catable_streams_stitch_like_brocatli(q):
    """BROTLI_PARAM_CATABLE (encode.rs:264-272, :2285-2333): the stream starts with its first two bytes as an uncompressed
    metablock, uses no static dictionary and ends with an empty last metablock, so the reference's BroCatli
    (src/concat/mod.rs, restated in tests/brocatli_ref.py) can splice it behind any other stream."""
    import brocatli_ref as bc
    a, b, c = golden_bytes("alice29.txt")[:90000], golden_bytes("asyoulik.txt")[:70000], golden_bytes("random_then_unicode")[:60000]
    sa = _framed(a, q, catable=True, magic_number=True)
    sb = _framed(b, q, catable=True)
    sc = _framed(c, q, catable=True, byte_align=True)
    for s, d in ((sa, a), (sb, b), (sc, c)):
        assert sys_decompress(s, len(d)) == d  # each is a complete stream on its own
        off = bc.first_metablock_aligned_offset(s)  # raises unless the stream starts with a metadata / uncompressed metablock
        assert off % 8 in (0, 1, 2, 3, 4, 5, 6, 7)
    # 4 window bits + 14 header bits of the metadata metablock, padded to 3 bytes; then e1 97 81 (catable), VERSION 1, size hint
    assert bytes(sa[3:6]) == b"\xe1\x97\x81" and sa[6] == 1
    assert sc[-1] == 3  # byte_align: padding metablock, then ISLAST + ISLASTEMPTY alone in the last byte
    whole = bc.concat([sa, sb, sc, _framed(b"", q, catable=True), sb])
    assert sys_decompress(whole, len(a) + 2 * len(b) + len(c)) == a + b + c + b
    with pytest.raises(bc.NotCraftedForConcatenation):  # a plain stream starts with a compressed metablock: the stitcher refuses it
        bc.concat([sa, _framed(b, q)])


def test_bare_and_appendable_streams_concatenate_by_memcpy():
    """bare_stream (encode.rs:277-282, :676, :1937): no window bits (with catable), no final metablock, byte aligned -- pieces
    are glued with memcpy behind a header-carrying first piece and closed with the single byte 0x03.  appendable + byte_align:
    strip that last byte and keep appending."""
    a, b, c = golden_bytes("alice29.txt")[:50000], golden_bytes("asyoulik.txt")[:40000], b"tail " * 2000
    head = _framed(a, 5, appendable=True, byte_align=True)
    assert head[-1] == 3 and sys_decompress(head, len(a)) == a
    mid = _framed(b, 5, catable=True, bare_stream=True)
    end = _framed(c, 9, catable=True, bare_stream=True)
    glued = head[:-1] + mid + end + b"\x03"
    assert sys_decompress(glued, len(a) + len(b) + len(c)) == a + b + c
    # bare without catable keeps the window bits: it is a first piece
    first = _framed(a, 5, bare_stream=True)
    assert sys_decompress(first + mid + b"\x03", len(a) + len(b)) == a + b


def test_framing_small_and_empty_inputs():
    import brocatli_ref as bc
    for d in (b"", b"x", b"xy", b"xyz", b"hello hello hello hello"):
        for kw in (dict(catable=True), dict(catable=True, magic_number=True), dict(appendable=True, byte_align=True),
                   dict(magic_number=True), dict(catable=True, byte_align=True)):
            s = _framed(d, 5, **kw)
            assert sys_decompress(s, max(1, len(d))) == d, (d, kw)
        s2 = bc.concat([_framed(b"abc", 5, catable=True), _framed(d, 5, catable=True)])
        assert sys_decompress(s2, 3 + len(d)) == b"abc" + d


def test_compress_multi_honours_framing():
    """CompressMulti with catable + magic_number: prologue of shard 0, trailer of the last shard; still one valid stream."""
    import rust_brotli_b200 as rb
    import brocatli_ref as bc
    d = golden_bytes("alice29.txt")
    c = rb.compress_multi(rb.BrotliEncoderParams(quality=5, lgwin=22, catable=True, magic_number=True, byte_align=True), d, 4)
    assert sys_decompress(c, len(d)) == d
    assert bytes(c[3:6]) == b"\xe1\x97\x81" and c[-1] == 3
    assert sys_decompress(bc.concat([c, c]), 2 * len(d)) == d + d


# ---- BASELINE.json configs at their full per-GPU sizes: size-independent properties (round trip, size bounds) ----

def test_config3_random10k_tiled_1gb(encoder):
    """configs[2]: random_org_10k.bin tiled to 1 GB, q5, lgwin 22 (period 10 000 B < window: the long-copy path; 42 chunks)."""
    from tools import datagen
    d = datagen.tiled(golden_bytes("random_org_10k.bin"), 1_000_000_000)
    c = encoder.compress(d, 5, 22)
    assert len(c) < 20_000  # one period of literals + one long copy per 4 MiB metablock
    assert hashlib.sha256(sys_decompress(c, len(d))).digest() == hashlib.sha256(d).digest()


def test_config3b_incompressible_256mb(encoder):
    """PCG bytes: every metablock is stored raw; size = input + a few bytes per metablock."""
    from tools import datagen
    d = datagen.pcg_random(256_000_000)
    c = encoder.compress(d, 5, 22)
    assert len(d) < len(c) <= len(d) + 8 * (len(d) // (4 << 20) + 2)
    assert sys_decompress(c, len(d)) == d


def test_config4_json_q9_one_shard_512mib():
    """configs[3]: JSON logs, q9, lgwin 22, compress_multi; one GPU's share (512 MiB) split into 8 byte-aligned shards that
    concatenate with memcpy (the reference needs BroCatli for that step)."""
    import rust_brotli_b200 as rb
    from tools import datagen
    d = datagen.json_logs(64_000_000) * 8
    d = d + d[:(512 << 20) - len(d)]
    assert len(d) == 512 << 20
    c = rb.compress_multi(rb.BrotliEncoderParams(quality=9, lgwin=22), d, 8)
    assert len(c) < 0.2 * len(d)
    assert hashlib.sha256(sys_decompress(c, len(d))).digest() == hashlib.sha256(d).digest()


def test_compress_multi_across_physical_gpus(encoder):
    """BrotliEncoderCompressMulti (src/ffi/multicompress/mod.rs:93; compress_multi threading/mod.rs:413) with 8 shards on a box
    with more than one GPU: one host thread per GPU, shards round-robin over the devices.  The stream must be the one a single
    GPU produces shard by shard (the kernels are deterministic), must decode, and more than one device must have worked."""
    import ctypes
    import rust_brotli_b200 as rb
    from tools import datagen
    L = rb.lib()
    L.b200_device_count.restype = ctypes.c_int
    ngpu = L.b200_device_count()
    if ngpu < 2:
        pytest.skip("needs at least 2 visible GPUs")
    d = datagen.json_logs(64_000_000) * 2
    c = rb.compress_multi(rb.BrotliEncoderParams(quality=9, lgwin=22), d, 8)
    L.b200_last_multi_device_mask.restype = ctypes.c_uint32
    mask = L.b200_last_multi_device_mask()
    assert bin(mask).count("1") == min(ngpu, 8), "shards ran on devices %s of %d" % (bin(mask), ngpu)
    assert hashlib.sha256(sys_decompress(c, len(d))).digest() == hashlib.sha256(d).digest()
    parts = []
    for i in range(8):
        a, b = i * len(d) // 8, (i + 1) * len(d) // 8
        win = (1 << 22) + 65536  # csrc/bro_capi.cu compress_span: the prefix handed over is re-based to one window (+ slack) in front
        lo = ((a - win) & ~4095) if a > win else 0
        parts.append(encoder.compress_range(d[lo:b], a - lo, b - a, 9, 22, i == 0, i == 7, True, size_hint=b - a))
    assert b"".join(parts) == c


def test_config5_quickfox_tiled_512mib_q11_lgwin24(encoder):
    """configs[4]: quickfox_repeated tiled to 512 MiB, quality 11 (all-matches + shortest-path parse + BrotliSplitBlock +
    clustered context maps on the device), lgwin 24.  libbrotlienc q11 needs 58 B for 16 MB of this input (one copy per
    metablock of <= 16 MiB); this path has 4 MiB metablocks of a few dozen bytes each (header + one copy)."""
    from tools import datagen
    d = datagen.tiled(golden_bytes("quickfox_repeated"), 512 << 20)
    c = encoder.compress(d, 11, 24)
    assert len(c) <= 64 + 64 * (len(d) // (4 << 20))
    assert hashlib.sha256(sys_decompress(c, len(d))).digest() == hashlib.sha256(d).digest()


@pytest.mark.parametrize("kind,q,bound", [("text", 10, 1.005), ("text", 11, 1.005), ("json", 10, 1.006), ("json", 11, 1.005)])
def test_hq_multi_metablock_equals_model_and_reference_size(encoder, model, kind, q, bound):
    """quality 10 / 11 on 6 MB of enwik-shaped text and of JSON logs (two metablocks, many parse units): bit identity with the CPU
    model, and size against libbrotlienc (the stated size reference for q >= 10, tests/golden/make_golden.py).  Measured with the
    three long-prefix candidate levels and, at q11, the first-pass statistics pooled over 64 KiB (bro_hq.cuh): text +0.24 % (q10) /
    +0.43 % (q11), JSON +0.47 % / +0.33 %; with the 4-byte bucket lists alone it was +1.2 / +1.5 % and +2.0 / +2.7 % (on the
    reference's own KAT file alice29 it is +0.1 %)."""
    import rust_brotli_b200 as rb
    from tools import datagen
    d = datagen.enwik_like(6_000_000) if kind == "text" else datagen.json_logs(6_000_000)
    c = encoder.compress(d, q, 22)
    assert sys_decompress(c, len(d)) == d
    assert c == model.compress(d, q, 22)[0]
    ref = len(sys_compress(d, q, 22))
    assert len(c) <= ref * bound, (len(c), ref)
    if kind == "text" and q == 10:  # the levels are what closes the gap: without them the same input is > 1 % larger
        encoder.set_option(rb._native.OPT_HQ_LEVELS, 0)
        try:
            c0 = encoder.compress(d, q, 22)
        finally:
            encoder.set_option(rb._native.OPT_HQ_LEVELS, 3)
        assert c0 == model.compress(d, q, 22, hq_levels=0)[0]
        assert len(c0) > ref * 1.01 > len(c)


def test_hq_options_equal_model(encoder, model):
    import rust_brotli_b200 as rb
    d = golden_bytes("asyoulik.txt") + golden_bytes("random_then_unicode")
    for opt, kw in ((rb._native.OPT_HQ_SPLIT, "hq_split"), (rb._native.OPT_DICT, "use_dict"), (rb._native.OPT_CTX_MODEL, "ctx_model")):
        encoder.set_option(opt, 0)
        try:
            c = encoder.compress(d, 10, 22)
        finally:
            encoder.set_option(opt, 1)
        assert sys_decompress(c, len(d)) == d
        assert c == model.compress(d, 10, 22, **{kw: 0})[0], kw
