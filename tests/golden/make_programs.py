"""Extracts the instruction tables of the reference's proving tests (basic/tests/test_prover.rs:190-402:
left_imm_ops_program, signed_inequality_program, loadfp_program) and the VM-state assertions that
follow them (test_prover.rs:490-625) into tests/golden/programs.json, so that the tests need no copy of the reference:
    python tests/golden/make_programs.py <reference checkout>"""
import json
import os
import re
import sys

SRC = os.path.join(sys.argv[1], "basic", "tests", "test_prover.rs")
OPC = {"Load32": 1, "Store32": 2, "Jal": 3, "Jalv": 4, "Beq": 5, "Bne": 6, "Imm32": 7, "Stop": 8, "LoadFp": 10, "Add32": 100, "Sub32": 101,
       "Lt32": 104, "Lte32": 115, "Slt32": 117, "Sle32": 118}
txt = open(SRC).read()
out = {}
for name in ["left_imm_ops_program", "signed_inequality_program", "loadfp_program"]:
    body = txt[txt.index("fn %s<" % name):]
    body = body[:body.index("\n}\n")]
    prog = []
    for m in re.finditer(r"opcode:\s*<(\w+)Instruction as Instruction<BasicMachine<Val>, Val>>::OPCODE,\s*operands:\s*(Operands\(\[([^\]]*)\]\)|Operands::default\(\))", body):
        ops = [0, 0, 0, 0, 0] if m.group(3) is None else [int(x.strip().replace("_", ""), 0) if not x.strip().startswith("-") else -int(x.strip()[1:].replace("_", ""), 0) for x in m.group(3).split(",") if x.strip()]
        prog.append([OPC[m.group(1)]] + ops)
    out[name] = {"program": prog}
for test, prog in [("prove_left_imm_ops", "left_imm_ops_program"), ("prove_signed_inequality", "signed_inequality_program"), ("prove_loadfp", "loadfp_program")]:
    body = txt[txt.index("fn %s()" % test):]
    body = body[:body.index("\n}\n")]
    cells = []
    for m in re.finditer(r"cells\.get\(&\(0x1000 \+ (\d+)\)\)\.unwrap\(\),\s*Word\(\[(\d+), (\d+), (\d+), (\d+),?\]\)", body):
        b = [int(m.group(i)) for i in range(2, 6)]
        cells.append([0x1000 + int(m.group(1)), (b[0] << 24) | (b[1] << 16) | (b[2] << 8) | b[3]])
    out[prog]["expected_cells"] = cells
json.dump(out, open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "programs.json"), "w"), indent=1)
print({k: (len(v["program"]), len(v["expected_cells"])) for k, v in out.items()})
