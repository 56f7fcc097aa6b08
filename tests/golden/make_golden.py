#!/usr/bin/env python3
"""Regenerate tests/golden/* from a checkout of the reference (dropbox/divans):

    python tests/golden/make_golden.py <reference checkout>

The reference holds no compressed golden vectors (SURVEY section 4), so the fixtures are made by feeding the
reference's own IR fixtures (testdata/*.ir, the input of src/bin/integration_test.rs:76-108) through the oracle
encoder; the EXPECTED OUTPUT side is pinned by the reference's raw testdata files (sha256 below), i.e. by real
reference data, not by the oracle.  Each entry: <name>.divans + an index line in golden.json.

reference_ir.json indexes what the tests take from the reference's IR fixtures without the reference at hand:
  samples   the first lines of each IR file (<name>.ir.xz) and the sha256 of the bytes they replay to, cut from the
            reference's raw file; the files themselves (up to 0.9 MB each) are too large to commit
  encodes   the stream the oracle encoder makes from a whole IR file; the tests rebuild the command list from the
            committed .divans fixture coded from that same IR and must reproduce this stream
brotli_transforms.json holds RFC 7932 dictionary words transformed by the system libbrotlicommon.so.1.
"""
import ctypes, hashlib, json, lzma, os, sys
import numpy as np
HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
from oracle import oracle_py as O

REF = os.path.join(sys.argv[1], "testdata") + os.sep
CASES = [
    # name, ir file, raw file, options
    ("alice29_ir", "alice29.ir", "alice29", dict()),
    ("alice29_priors_mix2", "alice29-priors.ir", "alice29", dict(dynamic_context_mixing=2)),
    ("alice29_priors_nocm", "alice29-priors.ir", "alice29", dict(dynamic_context_mixing=0, use_context_map=0)),
    ("alice29_q11_mix1", "alice29-q11.ir", "alice29", dict(dynamic_context_mixing=1)),
    ("asyoulik_ir_mix2", "asyoulik.ir", "asyoulik", dict(dynamic_context_mixing=2)),
    ("random_then_unicode_ir", "random_then_unicode.ir", "random_then_unicode", dict(dynamic_context_mixing=1)),
    ("truncated_dictionary", "ends_with_truncated_dictionary.ir", "ends_with_truncated_dictionary", dict()),
    ("alice29_literal_only", None, "alice29", dict()),
]
IR_SAMPLE_LINES = 4000      # covers every command kind each file uses (dict, prediction, ltype, ctype, dtype)
IR_SAMPLES = ["alice29", "asyoulik", "random_then_unicode", "ends_with_truncated_dictionary"]
IR_ENCODES = [
    # golden fixture coded from the IR, ir file, options of src/bin/integration_test.rs:235-236 / benchmark.rs:430-443
    ("alice29_ir", "alice29.ir", dict(dynamic_context_mixing=1)),
    ("random_then_unicode_ir", "random_then_unicode.ir", dict()),
]


def sha(b):
    return hashlib.sha256(b).hexdigest()


index = []
for name, ir, rawf, opts in CASES:
    raw = open(REF + rawf, "rb").read()
    o = O.options(**opts)
    if ir is None:
        enc = O.encode_raw(raw, o)
    else:
        enc = O.Commands.from_ir(open(REF + ir, "rb").read()).encode(o)
    rc, dec = O.decode(enc, out_cap=len(raw) + 64)
    assert rc == 0 and dec == raw, name
    open(os.path.join(HERE, name + ".divans"), "wb").write(enc)
    index.append(dict(name=name, source_ir=ir, source_raw=rawf, options=opts, raw_len=len(raw),
                      raw_sha256=hashlib.sha256(raw).hexdigest(), divans_len=len(enc), divans_sha256=hashlib.sha256(enc).hexdigest()))
    print(name, len(enc), len(raw))
json.dump(index, open(os.path.join(HERE, "golden.json"), "w"), indent=1)

samples = []
for rawf in IR_SAMPLES:
    lines = open(REF + rawf + ".ir", "rb").read().split(b"\n")
    n = min(IR_SAMPLE_LINES, len(lines) - 1)
    text = b"\n".join(lines[:n]) + b"\n"
    c = O.Commands.from_ir(text)
    rc, rec = c.recode(c.window or 22)
    raw = open(REF + rawf, "rb").read()
    assert rc == 0 and rec == raw[:len(rec)], rawf
    open(os.path.join(HERE, rawf + ".ir.xz"), "wb").write(lzma.compress(text, preset=9 | lzma.PRESET_EXTREME))
    samples.append(dict(name=rawf, source_ir="testdata/%s.ir" % rawf, lines=n, whole_file=n == len(lines) - 1, ir_sha256=sha(text),
                        raw_len=len(rec), raw_sha256=sha(rec)))
    print(rawf, "sample", n, "lines ->", len(rec), "bytes")
encodes = []
for gname, ir, opts in IR_ENCODES:
    enc = O.Commands.from_ir(open(REF + ir, "rb").read()).encode(O.options(**opts))
    rc, _, cmds = O.decode_cmds(open(os.path.join(HERE, gname + ".divans"), "rb").read())
    assert rc == 0 and cmds.encode(O.options(**opts)) == enc, gname
    encodes.append(dict(golden=gname, source_ir="testdata/" + ir, options=opts, divans_len=len(enc), divans_sha256=sha(enc)))
json.dump(dict(samples=samples, encodes=encodes), open(os.path.join(HERE, "reference_ir.json"), "w"), indent=1)

# RFC 7932 transforms of random dictionary words by libbrotlicommon's BrotliTransformDictionaryWord
lib = ctypes.CDLL("libbrotlicommon.so.1")
lib.BrotliGetTransforms.restype = ctypes.c_void_p
lib.BrotliGetDictionary.restype = ctypes.c_void_p
lib.BrotliTransformDictionaryWord.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p, ctypes.c_int]
lib.BrotliTransformDictionaryWord.restype = ctypes.c_int


class BD(ctypes.Structure):
    _fields_ = [("sb", ctypes.c_uint8 * 32), ("off", ctypes.c_uint32 * 32), ("n", ctypes.c_size_t), ("data", ctypes.POINTER(ctypes.c_uint8))]


d = ctypes.cast(lib.BrotliGetDictionary(), ctypes.POINTER(BD)).contents
tr = lib.BrotliGetTransforms()
rng = np.random.default_rng(7)
vectors = []
for _ in range(600):
    ws = int(rng.integers(4, 25))
    wid = int(rng.integers(0, 1 << d.sb[ws]))
    t = int(rng.integers(0, 121))
    out = np.zeros(64, np.uint8)
    n = lib.BrotliTransformDictionaryWord(out.ctypes.data, ctypes.addressof(d.data.contents) + d.off[ws] + wid * ws, ws, tr, t)
    vectors.append([ws, wid, t, out[:n].tobytes().hex()])
json.dump(dict(source="libbrotlicommon.so.1 BrotliTransformDictionaryWord(word_size, word_id, transform)", vectors=vectors),
          open(os.path.join(HERE, "brotli_transforms.json"), "w"), separators=(",", ":"))
