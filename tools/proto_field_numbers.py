"""Record the field / enum numbers of apache/datafusion-comet's plan IR as tests/golden/proto_field_numbers.json.

usage: python tools/proto_field_numbers.py <datafusion-comet checkout>/native/proto/src/proto [out.json]

The hand-written encoder (comet_b200/proto.py) and decoder (csrc/plan.cpp) must use the same numbers as the .proto files
(tests/test_proto.py checks them against this record).  Rerun when moving to another datafusion-comet release."""
import json
import os
import re
import sys

FILES = ("expr", "operator", "types", "literal", "partitioning")


def parse_proto(path):
    """{message_or_enum: {field_name: number}} with nested messages flattened by simple name; oneof members belong to the
    enclosing message."""
    txt = re.sub(r"//[^\n]*", "", open(path).read())
    out = {}
    stack = []
    for tok in re.finditer(r"(message|enum|oneof)\s+(\w+)\s*\{|\}|(?:repeated\s+|optional\s+)?[\w.<>, ]+?\s+(\w+)\s*=\s*(\d+)\s*(?:\[[^\]]*\])?;|(\w+)\s*=\s*(-?\d+)\s*;", txt):
        if tok.group(1):
            stack.append((tok.group(1), tok.group(2)))
            if tok.group(1) != "oneof":
                out.setdefault(tok.group(2), {})
        elif tok.group(0) == "}":
            if stack:
                stack.pop()
        else:
            name, num = (tok.group(3), tok.group(4)) if tok.group(3) else (tok.group(5), tok.group(6))
            owner = next((n for k, n in reversed(stack) if k != "oneof"), None)
            if owner:
                out[owner][name] = int(num)
    return out


def main():
    src = sys.argv[1]
    dst = sys.argv[2] if len(sys.argv) > 2 else os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))),
                                                             "tests", "golden", "proto_field_numbers.json")
    rec = {f: parse_proto(os.path.join(src, f + ".proto")) for f in FILES}
    with open(dst, "w") as f:
        json.dump(rec, f, indent=1, sort_keys=True)
        f.write("\n")


if __name__ == "__main__":
    main()
