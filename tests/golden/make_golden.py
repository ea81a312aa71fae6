"""Generates tests/golden/reference_tables.json from the reference checkout (run in the build container only).

The reference has no byte-level golden vectors for the hot path (SURVEY.md §8c); what it does hold are data tables and
constants that the oracle re-derives from formulas. This script extracts them verbatim so that the CPU tests can pin
the oracle's derivations without reading /root/reference at test time.
"""
import json
import os
import re
import sys

REF = sys.argv[1] if len(sys.argv) > 1 else "/root/reference/v2"


def go_array(text, name):
    m = re.search(name + r"\s*=\s*\[[^\]]*\](?:\[[^\]]*\])?\w+\s*\{", text)
    assert m, name
    i = m.end()
    depth = 1
    j = i
    while depth:
        c = text[j]
        depth += c == "{"
        depth -= c == "}"
        j += 1
    body = re.sub(r"//[^\n]*", "", text[i:j - 1])
    return [int(x, 0) for x in re.findall(r"0x[0-9a-fA-F]+|\d+", body)]


def main():
    out = {}
    eg = open(os.path.join(REF, "entropy/ExpGolombCodec.go")).read()
    vals = go_array(eg, "_EXPG_VALUES")
    assert len(vals) == 512
    out["expg_unsigned"] = vals[:256]
    out["expg_signed"] = vals[256:]
    gl = open(os.path.join(REF, "internal/Global.go")).read()
    out["log2_4096"] = go_array(gl, "LOG2_4096")
    out["log2"] = go_array(gl, r"LOG2")
    cs = open(os.path.join(REF, "io/CompressedStream.go")).read()
    out["bitstream_type"] = int(re.search(r"_BITSTREAM_TYPE\s*=\s*(0x[0-9A-Fa-f]+)", cs).group(1), 16)
    out["bitstream_version"] = int(re.search(r"_BITSTREAM_FORMAT_VERSION\s*=\s*(\d+)", cs).group(1))
    ef = open(os.path.join(REF, "entropy/EntropyCodecFactory.go")).read()
    out["entropy_ids"] = {m.group(1): int(m.group(2)) for m in re.finditer(r"(\w+)_TYPE\s*=\s*uint32\((\d+)\)", ef)}
    tf = open(os.path.join(REF, "transform/Factory.go")).read()
    out["transform_ids"] = {m.group(1): int(m.group(2)) for m in re.finditer(r"(\w+)_TYPE\s*=\s*uint64\((\d+)\)", tf)}
    # values of the reference's own varint size test (entropy/Entropy_test.go:54-69); expected size = 1 + #(7-bit groups beyond the first)
    out["varint_values"] = [0, 1, 127, 128, 255, 16384, (1 << 21) - 1, 1 << 21, (1 << 28) - 1, 1 << 28, 0xFFFFFFFF]
    with open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "reference_tables.json"), "w") as f:
        json.dump(out, f, indent=0)
    print({k: (len(v) if hasattr(v, "__len__") else v) for k, v in out.items()})
    # TEXT's static dictionary (transform/TextCodec.go, _TC_DICT_EN_1024), a constant of the format that the library and the oracle embed
    # (kanzi-go_b200/gen_text_dict.py, oracle/gen_text_dict.py): one word per line, letters only, as createDictionary reads it
    tc = open(os.path.join(REF, "transform/TextCodec.go"), encoding="utf-8").read()
    letters = "".join(c for c in re.search(r"_TC_DICT_EN_1024\s*=\s*\[\]byte\(`([^`]*)`\)", tc).group(1) if c.isascii() and c.isalpha())
    words = re.findall(r"[A-Z][a-z]*", letters)
    assert len(words) == 1024 and "".join(words) == letters
    with open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "text_dict_en_1024.txt"), "w") as f:
        f.write("\n".join(words) + "\n")
    print({"text_dict_en_1024": len(words)})


if __name__ == "__main__":
    main()
