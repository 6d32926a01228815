"""Extract the exported `fit` / `decisionFunction` signatures of the reference procs the Nim host layer (nim/*.nim)
replaces, into tests/golden/nim_signatures.json.  Needs a checkout of the reference (nimfm); the JSON is committed so
the CPU test does not need the reference tree.

    python tests/golden/make_nim_signatures.py <nimfm checkout>/src/nimfm
"""
import json
import os
import re
import sys

FILES = ["optimizer/cd.nim", "optimizer/minibatch_psgd.nim", "optimizer/adagrad.nim", "optimizer/adagrad_multi.nim",
         "optimizer/adagrad_ffm.nim", "optimizer/adagrad_ffm_multi.nim", "optimizer/sgd.nim", "optimizer/sgd_multi.nim",
         "optimizer/sgd_ffm.nim", "optimizer/sgd_ffm_multi.nim", "model/factorization_machine.nim",
         "model/field_aware_factorization_machine.nim"]
NAMES = ("fit", "decisionFunction")


def signatures(text):
    """every exported proc NAME*...(...)[: ret] = header, whitespace-normalised, keyed in order of appearance"""
    out = []
    for m in re.finditer(r"^proc (%s)\*" % "|".join(NAMES), text, flags=re.M):
        depth, i = 0, m.start()
        # the header ends at the '=' that follows the balanced parameter list (and an optional return type)
        j = text.index("(", m.end() - 1) if text[m.end()] in "[(" else m.end()
        k = j
        seen_paren = False
        while k < len(text):
            c = text[k]
            if c == "(":
                depth += 1
                seen_paren = True
            elif c == ")":
                depth -= 1
            elif c == "=" and depth == 0 and seen_paren and text[k + 1] != "=" and text[k - 1] not in "<>!=" \
                    and text[k + 1] != ">":
                break
            k += 1
        out.append(re.sub(r"\s+", " ", text[i:k]).strip())
    return out


def main(ref):
    table = {}
    for f in FILES:
        table[f] = signatures(open(os.path.join(ref, f)).read())
    here = os.path.dirname(os.path.abspath(__file__))
    json.dump(table, open(os.path.join(here, "nim_signatures.json"), "w"), indent=1)
    for f, sigs in table.items():
        for s in sigs:
            print(f, "::", s)


if __name__ == "__main__":
    main(sys.argv[1])
