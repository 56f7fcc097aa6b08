#!/usr/bin/env python3
"""Extract the one compressed stream the reference tree holds: `_example_dv_file`, wasm/wasm.html:98-107 (113 bytes,
written by the reference's own Rust encoder; its trailer CRC32C is valid):

    python tests/golden/extract_wasm_vector.py <reference checkout>

writes tests/golden/ref_wasm_example.divans.  The expected plaintext is not in the reference tree; it
is what the stream decodes to under model revision WASM_2018 (oracle/divans_oracle.h) -- human-readable English with
a valid CRC -- and is recorded in ref_wasm_example.json for the GPU tests."""
import hashlib, json, os, re, sys
HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
text = open(os.path.join(sys.argv[1], "wasm", "wasm.html")).read()
m = re.search(r"_example_dv_file\s*=\s*\[(.*?)\]", text, re.S)
vec = bytes(int(x, 16) for x in re.findall(r"0x([0-9a-fA-F]{2})", m.group(1)))
assert len(vec) == 113 and vec[:4] == bytes([0xff, 0xe5, 0x8c, 0x9f]) and vec[-4:] == b"ans~"
open(os.path.join(HERE, "ref_wasm_example.divans"), "wb").write(vec)
from oracle import oracle_py as O
assert O.crc32c(vec[:-8]) == int.from_bytes(vec[-8:-4], "little")
rc, plain, cmds = O.decode_cmds(vec, model_rev=O.MODEL_WASM_2018)
assert rc == 0, rc
json.dump(dict(source="wasm/wasm.html:98-107", divans_len=len(vec), divans_sha256=hashlib.sha256(vec).hexdigest(),
               model_rev="WASM_2018", plain_len=len(plain), plain_sha256=hashlib.sha256(plain).hexdigest(),
               plain_text=plain.decode("ascii"), n_cmds=int(cmds.n_cmds)),
          open(os.path.join(HERE, "ref_wasm_example.json"), "w"), indent=1)
print(len(vec), len(plain), plain[:48])
