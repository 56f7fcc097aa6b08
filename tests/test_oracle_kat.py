"""CPU tests: pin the oracle (oracle/divans_oracle.c) against every known-answer test the reference holds for the
divANS path (SURVEY 8c).  Reference citations name the test that carries the vector."""
import ctypes
import hashlib
import json
import lzma
import os

import numpy as np

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def test_crc32c_known_answers(oracle):
    # reference src/codec/crc32.rs:90-115
    assert oracle.crc32c(b"") == 0
    assert oracle.crc32c(b"123456789") == 0xE3069283
    assert oracle.crc32c(b"6789", oracle.crc32c(b"12345")) == 0xE3069283
    q = b"The quick brown fox jumps over the lazy dog"
    assert oracle.crc32c(q) == 0x22620404
    assert oracle.crc32c(q[18:], oracle.crc32c(q[:18])) == 0x22620404


def test_fast_divide_known_answers(oracle):
    # reference src/probability/numeric.rs:74-86
    nums = [3032127, 5049117, 16427165, 23282359, 35903174, 132971515, 163159927, 343856773, 935221996, 1829347323]
    denoms = [115, 248, 267, 764, 1337, 4005, 4965, 9846, 24693, 31604]
    L = oracle.lib()
    for n in nums:
        for d in denoms:
            assert L.dvo_fast_divide(n, d) == n // d
    # the LUT generator's exhaustive claim (make_div_lut.rs:37-39), sampled
    rng = np.random.default_rng(1)
    for d in rng.integers(1, 32768, 200):
        for c in rng.integers(0, 65536, 50):
            assert L.dvo_fast_divide(int(c) << 15, int(d)) == (int(c) << 15) // int(d)


def test_f8_speed_codec(oracle):
    # reference src/probability/interface.rs:586-617
    L = oracle.lib()
    for v in [0, 1, 2, 3, 4, 5, 6, 7, 8, 10, 12, 16, 24, 32, 48, 64, 96, 768, 1280, 1536, 1664]:
        assert L.dvo_u8_to_speed(L.dvo_speed_to_u8(v)) == v


def test_mux_decode_vector(oracle):
    # reference src/test_mux.rs:1192-1207 (41-byte literal vector)
    v = bytes([0x0, 0xf, 0x0, 0x75, 0x98, 0x10, 0x40, 0x2, 0x5, 0x8, 0x0, 0x4f, 0x85, 0x92, 0x18, 0x40, 0x80, 0x0, 0x0,
               0x1, 0xf, 0x0, 0x1, 0x2a, 0x0, 0x1, 0x8, 0x0, 0x0, 0x0, 0x1, 0x42, 0x0, 0x1, 0x8, 0x0, 0x0, 0x0, 0xff, 0xfe, 0xff])
    cmd, lit = oracle.demux(bytes(16) + v)
    assert cmd == v[3:19] and lit == v[22:38]


def test_mux_roundtrip_record_shapes(oracle):
    # framing produced at close (mux.rs:55-78,478-561): 65536-byte fixed records then one variable record
    L = oracle.lib()
    for n in [1, 15, 4095, 4096, 4097, 16384, 65535, 65536, 65537, 200000]:
        data = np.random.default_rng(n).integers(0, 256, n).astype(np.uint8)
        out = np.zeros(n + 64, np.uint8)
        m = L.dvo_mux_single(1, data.ctypes.data, n, out.ctypes.data, out.size)
        cmd, lit = oracle.demux(bytes(16) + out[:m].tobytes())
        assert cmd == b"" and lit == data.tobytes()
        assert out[m - 3:m].tobytes() == b"\xff\xfe\xff"


def test_dictionary_words(oracle):
    # reference src/cmd_to_raw/test.rs:49-152: word_size 22, ids 0..4, transform 1 then transform 4
    L = oracle.lib()
    exp1 = bytes([100, 101, 115, 99, 114, 105, 112, 116, 105, 111, 110, 34, 32, 99, 111, 110, 116, 101, 110, 116, 61, 34, 32, 100,
                  111, 99, 117, 109, 101, 110, 116] +
                 [46, 108, 111, 99, 97, 116, 105, 111, 110, 46, 112, 114, 111, 116, 32, 46, 103, 101, 116, 69, 108, 101, 109, 101,
                  110, 116, 115, 66, 121, 84, 97] +
                 [103, 78, 97, 109, 101, 40, 32, 60, 33, 68, 79, 67, 84, 89, 80, 69, 32, 104, 116, 109, 108, 62, 10, 60, 104, 116,
                  109, 108] +
                 [32, 32, 60, 109, 101, 116, 97, 32, 99, 104, 97, 114, 115, 101, 116, 61, 34, 117, 116, 102, 45, 56, 34, 62, 32])
    for transform, first in [(1, exp1), (4, bytes([68]) + exp1[1:23] + bytes([68]) + exp1[24:])]:
        got = b""
        for wid in range(5):
            buf = np.zeros(64, np.uint8)
            n = L.dvo_dict_word(22, wid, transform, buf.ctypes.data)
            assert n == 23
            got += buf[:n].tobytes()
        assert got == first


def test_transform_matches_system_brotli(oracle):
    # cross-check our RFC 7932 transform against libbrotlicommon's BrotliTransformDictionaryWord: 600 random
    # (word size, word id, transform) triples and the words it made of them (tests/golden/make_golden.py)
    vectors = json.load(open(os.path.join(GOLD, "brotli_transforms.json")))["vectors"]
    assert len(vectors) == 600
    L = oracle.lib()
    for ws, wid, t, ref in vectors:
        mine = np.zeros(64, np.uint8)
        n = L.dvo_dict_word(ws, wid, t, mine.ctypes.data)
        assert mine[:n].tobytes().hex() == ref, (ws, wid, t)


def _cdf(oracle, vals=None):
    c = oracle.Cdf16()
    oracle.lib().dvo_cdf_default(ctypes.byref(c))
    if vals is not None:
        for i, v in enumerate(vals):
            c.c[i] = v
    return c


def test_cdf_invariants(oracle):
    # reference src/probability/common_tests.rs:4-103: monotone ranges, search covers all 32768 offsets, non-zero pdf
    L = oracle.lib()
    rng = np.random.default_rng(3)
    c = _cdf(oracle)
    assert list(c.c) == [4 * (i + 1) for i in range(16)]
    for step in range(3000):
        sym = int(rng.integers(0, 16)) if step % 3 else int(rng.integers(0, 3))
        L.dvo_cdf_blend(ctypes.byref(c), sym, oracle.Speed(int(rng.choice([16, 32, 48, 96, 128, 384])), 16384))
        vals = list(c.c)
        assert all(b > a for a, b in zip(vals, vals[1:])) and vals[0] > 0 and vals[15] < 32768
    # every cdf_offset maps into the [start, start+freq) of the symbol it decodes to, ranges are disjoint and ordered
    start, freq = ctypes.c_int16(), ctypes.c_int16()
    prev_end, prev_sym = 0, 0
    for off in range(0, 32768, 7):
        sym = L.dvo_cdf_lookup(ctypes.byref(c), off, ctypes.byref(start), ctypes.byref(freq))
        assert freq.value > 0 and start.value >= 0
        s2, f2 = ctypes.c_int16(), ctypes.c_int16()
        L.dvo_cdf_sym_start_freq(ctypes.byref(c), sym, ctypes.byref(s2), ctypes.byref(f2))
        assert (s2.value, f2.value) == (start.value, freq.value)
        assert sym >= prev_sym
        prev_sym = sym


def test_average_is_between(oracle):
    L = oracle.lib()
    a, b, out = _cdf(oracle), _cdf(oracle), _cdf(oracle)
    for _ in range(200):
        L.dvo_cdf_blend(ctypes.byref(a), 3, oracle.Speed(128, 16384))
        L.dvo_cdf_blend(ctypes.byref(b), 11, oracle.Speed(48, 4096))
    for w in [0, 1 << 14, 1 << 15]:
        L.dvo_cdf_average(ctypes.byref(a), ctypes.byref(b), w, ctypes.byref(out))
        vals = list(out.c)
        assert all(y >= x for x, y in zip(vals, vals[1:]))


def test_golden_fixtures_decode_to_reference_data(oracle, golden):
    # expected side = sha256 of the reference's raw testdata files (tests/golden/make_golden.py)
    for e in golden:
        enc = open(e["path"], "rb").read()
        assert hashlib.sha256(enc).hexdigest() == e["divans_sha256"]
        rc, dec = oracle.decode(enc, out_cap=e["raw_len"] + 64)
        assert rc == 0 and len(dec) == e["raw_len"]
        assert hashlib.sha256(dec).hexdigest() == e["raw_sha256"], e["name"]


def test_encoder_is_deterministic_against_golden(oracle, golden):
    # re-encoding the literal-only fixture input must reproduce the committed stream byte for byte
    e = [g for g in golden if g["name"] == "alice29_literal_only"][0]
    enc = open(e["path"], "rb").read()
    rc, raw = oracle.decode(enc, out_cap=e["raw_len"] + 64)
    assert rc == 0 and oracle.encode_raw(raw) == enc


def _reference_ir():
    return json.load(open(os.path.join(GOLD, "reference_ir.json")))


def _golden_raw(oracle, golden, name):
    # the reference's raw testdata file, as the committed fixture coded from it decodes (sha256 pinned in golden.json)
    e = [g for g in golden if g["name"] == name][0]
    rc, raw = oracle.decode(open(e["path"], "rb").read(), out_cap=e["raw_len"] + 64)
    assert rc == 0 and hashlib.sha256(raw).hexdigest() == e["raw_sha256"]
    return raw


def test_ir_fixtures_recode_to_raw(oracle):
    # reference src/bin/integration_test.rs:76-108, on the first 4000 lines of each IR file (the whole file for
    # ends_with_truncated_dictionary): they replay to the first bytes of the reference's raw file
    samples = _reference_ir()["samples"]
    assert [s["name"] for s in samples] == ["alice29", "asyoulik", "random_then_unicode", "ends_with_truncated_dictionary"]
    for s in samples:
        text = lzma.decompress(open(os.path.join(GOLD, s["name"] + ".ir.xz"), "rb").read())
        assert hashlib.sha256(text).hexdigest() == s["ir_sha256"], s["name"]
        c = oracle.Commands.from_ir(text)
        rc, rec = c.recode(c.window or 22)
        assert rc == 0 and len(rec) == s["raw_len"] and hashlib.sha256(rec).hexdigest() == s["raw_sha256"], s["name"]


def test_ratio_ceilings(oracle, golden):
    # reference src/bin/integration_test.rs:235-236 (alice29 <= 0.34 with brotli commands, <= 0.46 literal-only),
    # src/bin/benchmark.rs:430-443 (random_then_unicode IR <= 0.6).  The command list of a whole IR file is the one the
    # committed fixture coded from it carries; re-encoded, it must give the stream the reference's IR file gives.
    raw = _golden_raw(oracle, golden, "alice29_literal_only")
    assert len(oracle.encode_raw(raw)) / len(raw) <= 0.46
    encodes = {e["source_ir"]: e for e in _reference_ir()["encodes"]}
    for ir, raw_name, ceiling in [("alice29.ir", "alice29_literal_only", 0.34), ("random_then_unicode.ir", "random_then_unicode_ir", 0.6)]:
        e = encodes["testdata/" + ir]
        raw = _golden_raw(oracle, golden, raw_name)
        rc, _, c = oracle.decode_cmds(open(os.path.join(GOLD, e["golden"] + ".divans"), "rb").read())
        assert rc == 0
        enc = c.encode(oracle.options(**e["options"]))
        assert len(enc) == e["divans_len"] and hashlib.sha256(enc).hexdigest() == e["divans_sha256"], ir
        assert len(enc) / len(raw) <= ceiling, ir


def test_roundtrip_edge_cases(oracle):
    # empty, 1 byte, around the 8-byte last_8_literals quirk, 15/16-byte literal lengths, chunk boundary 65536 symbols
    rng = np.random.default_rng(5)
    for n in [0, 1, 2, 7, 8, 9, 14, 15, 16, 17, 255, 32767, 32768, 32769, 70001]:
        raw = rng.integers(97, 123, n).astype(np.uint8).tobytes()
        for win in [10, 22]:
            enc = oracle.encode_raw(raw, oracle.options(window_size=win))
            rc, dec = oracle.decode(enc, out_cap=n + 64)
            assert rc == 0 and dec == raw, (n, win)


def test_truncation_and_corruption_are_detected(oracle):
    raw = bytes(range(256)) * 20
    enc = oracle.encode_raw(raw)
    for cut in [0, 5, 16, 40, len(enc) - 9, len(enc) - 1]:
        rc, _ = oracle.decode(enc[:cut], out_cap=len(raw) + 64)
        assert rc == oracle.NEEDS_MORE_INPUT
    bad = bytearray(enc)
    bad[len(bad) // 2] ^= 0x40
    rc, _ = oracle.decode(bytes(bad), out_cap=len(raw) + 64)
    assert rc != oracle.SUCCESS            # garbage symbols (underflow / bad command) or, at the latest, the CRC32C trailer
    rc, dec = oracle.decode(bytes(bad), out_cap=len(raw) + 64, skip_crc=True)
    assert rc in (oracle.SUCCESS, oracle.FAILURE, oracle.NEEDS_MORE_INPUT, oracle.NEEDS_MORE_OUTPUT)
    rc, _ = oracle.decode(enc, out_cap=100)
    assert rc == oracle.NEEDS_MORE_OUTPUT


def test_lz77_roundtrip_and_window_wrap(oracle):
    rng = np.random.default_rng(9)
    base = rng.integers(97, 105, 3000).astype(np.uint8).tobytes()
    raw = base * 30                      # 90 kB of repeats: long copies, output longer than a 2^10 window
    for win in [10, 12, 16, 22]:
        c = oracle.Commands.lz77(raw, window=win)
        enc = c.encode(oracle.options(window_size=win, dynamic_context_mixing=2))
        rc, dec = oracle.decode(enc, out_cap=len(raw) + 64)
        assert rc == 0 and dec == raw


def test_random_ir_roundtrip(oracle):
    # encode(IR) -> decode must equal the ring-buffer replay of the same IR, for random valid command mixes
    import sys, os
    sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
    import irfuzz
    from divans_b200 import synth
    text = synth.text_corpus(1 << 16)
    for seed in range(24):
        win = [10, 14, 16, 22][seed % 4]
        c = oracle.Commands.from_ir(irfuzz.random_ir(oracle, seed, n_cmds=120, window=win, text=text))
        rc, raw = c.recode(win)
        assert rc == 0
        o = oracle.options(window_size=win, dynamic_context_mixing=seed % 3, use_context_map=0 if seed % 7 == 3 else 1,
                           force_stride=9 if seed % 5 else 3, prior_depth=seed % 4)
        enc = c.encode(o)
        rc, dec = oracle.decode(enc, out_cap=len(raw) + 64)
        assert rc == 0 and dec == raw, seed


# ---------------------------------------------------------------------------------------------------------------
# The one compressed stream the reference tree holds (wasm/wasm.html:98-107): whole-bitstream pin of the oracle.
# ---------------------------------------------------------------------------------------------------------------
def _wasm_vector():
    vec = open(os.path.join(GOLD, "ref_wasm_example.divans"), "rb").read()
    meta = json.load(open(os.path.join(GOLD, "ref_wasm_example.json")))
    return vec, meta


def test_reference_held_stream_fixture_is_the_reference_bytes():
    # the committed fixture equals what wasm/wasm.html holds: its sha256 was taken from that array when it was extracted
    # (tests/golden/extract_wasm_vector.py)
    vec, meta = _wasm_vector()
    assert len(vec) == 113 and hashlib.sha256(vec).hexdigest() == meta["divans_sha256"]
    assert meta["divans_sha256"] == "1aa983e906e5dc781f21c25baea8992c37b3fa12aa4ae45a4d847c43c476869a"


def test_reference_held_stream_decodes_under_its_model_revision(oracle):
    vec, meta = _wasm_vector()
    # container: magic, window 22, two records, EOF marker, CRC32C(header..marker) LE32, "ans~"
    assert vec[:6] == bytes([0xff, 0xe5, 0x8c, 0x9f, 0x00, 0x16]) and vec[-4:] == b"ans~"
    assert oracle.crc32c(vec[:-8]) == int.from_bytes(vec[-8:-4], "little")
    cmd, lit = oracle.demux(vec)
    assert (len(cmd), len(lit)) == (44, 36)
    rc, plain, cmds = oracle.decode_cmds(vec, model_rev=oracle.MODEL_WASM_2018)   # CRC checked (skip_crc=False)
    assert rc == oracle.SUCCESS
    assert plain == b"It snowed, rained, and hailed the same morning.\n" * 7
    assert plain.decode("ascii") == meta["plain_text"] and hashlib.sha256(plain).hexdigest() == meta["plain_sha256"]
    # 9 commands: PredictionMode (UTF8, empty context maps, 8192 x mixing value 4), a literal block switch, literals of
    # 15 / 11 / 2 bytes, copy(distance 8, 4 bytes), two dictionary words, copy(distance 48, 288 bytes): rANS, CDF arithmetic,
    # command / literal / copy / dictionary / block-switch coding, the RFC 7932 dictionary, mux framing and CRC32C are
    # all exercised by this stream.
    assert cmds.n_cmds == meta["n_cmds"] == 9 and cmds.window == 22


def test_reference_held_stream_is_reproduced_by_the_encoder(oracle):
    # the encoder half: same commands, same options (use_context_map=0 -> mixing values 4, no maps; mixing nibble 0)
    # -> the reference encoder's own 113 bytes, byte for byte (both rANS payloads, record framing, CRC)
    vec, _ = _wasm_vector()
    rc, plain, cmds = oracle.decode_cmds(vec, model_rev=oracle.MODEL_WASM_2018)
    assert rc == 0
    enc = cmds.encode(oracle.options(window_size=22, use_context_map=0, dynamic_context_mixing=0, model_rev=oracle.MODEL_WASM_2018))
    assert enc == vec


def test_reference_held_stream_version_skew_is_exactly_two_constructs(oracle):
    # Under the model of the mounted source tree the stream does NOT decode: command nibbles 1..20 agree (PredictionMode,
    # UTF8, mixing 0, depth 0, MUD x4), nibble 21 (first context-map mnemonic, codec/context_map.rs:273) is coded with
    # PredictionModePriorType::Mnemonic's own fresh slot today (codec/priors.rs:130) -- the stream needs the slot shared by
    # DynamicContextMixingSpeed/PriorDepth/ContextMapSpeedPalette[0]; and mixing values >= 256 use value[i-256] as prior
    # today (context_map.rs:395-399) -- the stream uses slot 16 throughout.
    vec, _ = _wasm_vector()
    rc, plain = oracle.decode(vec)
    assert rc == oracle.NEEDS_MORE_INPUT and plain == b""
    # the same commands under today's model round-trip, and differ from the 2018 stream only in the command coder's bytes
    rc, plain, cmds = oracle.decode_cmds(vec, model_rev=oracle.MODEL_WASM_2018)
    now = cmds.encode(oracle.options(window_size=22, use_context_map=0, dynamic_context_mixing=0))
    rc2, plain2 = oracle.decode(now)
    assert rc2 == 0 and plain2 == plain
    assert oracle.demux(now)[1] == oracle.demux(vec)[1]      # literal coder payload: identical
    assert oracle.demux(now)[0] != oracle.demux(vec)[0]      # command coder payload: the PredictionMode priors differ
