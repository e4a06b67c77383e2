"""Writes the SASS of the hot loops to profiles/sass/ (cuobjdump of the objects build.py leaves under capycrypt_b200/_lib).
usage: python profiles/extract_sass.py
  keccak_round_x2.sass     the two-round loop body of sha3_short_kernel<17, 8> (headline, bitsliced): 248 LOP3 + 104 SHFL
  keccak_pair_round.sass   one iteration (4 rounds) of the split-lane permutation inside sponge_tiered_kernel<9>
  keccak_warp_round.sass   the first rounds of the unrolled one-lane-per-thread permutation
  fe_mul.sass / fe_sqr.sass the out-of-line field multiplication / squaring of ed448_var.cu
  pair_prefetch_before_permutation.sass   the pair tier's step: predicated loads of the next block, then the permutation
  chain_ticket_and_wait.sass / chain_report.sass   sponge_chain_kernel<17>: ticket, dependency wait, completion report
  opcode_histograms.txt    instruction mix per kernel
"""
import collections
import glob
import os
import re
import subprocess

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
OBJ = sorted(glob.glob(os.path.join(ROOT, "capycrypt_b200", "_lib", "obj_*")), key=os.path.getmtime)[-1]
OUT = os.path.join(ROOT, "profiles", "sass")
os.makedirs(OUT, exist_ok=True)


def functions(obj):
    txt = subprocess.run(["cuobjdump", "-sass", obj], capture_output=True, text=True).stdout
    res = {}
    for part in re.split(r"\n\s+Function : ", txt)[1:]:
        name, body = part.split("\n", 1)
        ins = []
        for line in body.split("\n"):
            m = re.match(r"\s+/\*([0-9a-f]{4,5})\*/\s+(.*?);", line)
            if m:
                ins.append((int(m.group(1), 16), m.group(2).strip()))
        res[name.strip()] = ins
    return res


def opcode(t):
    t = re.sub(r"^@!?U?P\d+\s+", "", t)
    op = t.split()[0]
    base = op.split(".")[0]
    if base == "IMAD" and ".WIDE" in op:
        return "IMAD.WIDE"
    return base


def loops(ins):
    addr = {a: i for i, (a, _) in enumerate(ins)}
    for i, (a, t) in enumerate(ins):
        if re.match(r"(@!?U?P\d+\s+)?BRA", t):
            m = re.search(r"0x([0-9a-f]+)", t)
            if m and int(m.group(1), 16) < a and int(m.group(1), 16) in addr:
                yield addr[int(m.group(1), 16)], i


def dump(path, header, ins):
    with open(path, "w") as f:
        f.write("// " + header + "\n")
        for a, t in ins:
            f.write(f"/*{a:05x}*/  {t} ;\n")


sha3 = functions(os.path.join(OBJ, "sha3_api.o"))
var = functions(os.path.join(OBJ, "ed448_var.o"))
hist = []
for name, ins in list(sha3.items()) + list(functions(os.path.join(OBJ, "ed448_fixed.o")).items()) + list(var.items()):
    c = collections.Counter(opcode(t) for _, t in ins)
    hist.append(f"{name[:90]}\n    {len(ins)} instructions: " + ", ".join(f"{k} {v}" for k, v in c.most_common(12)))
open(os.path.join(OUT, "opcode_histograms.txt"), "w").write("\n".join(hist) + "\n")

short = next(v for k, v in sha3.items() if "sha3_short_kernelILi17ELi8E" in k)
s, e = max(loops(short), key=lambda se: se[1] - se[0])
dump(os.path.join(OUT, "keccak_round_x2.sass"), "sha3_short_kernel<17, 8>: loop body = two Keccak-f rounds", short[s:e + 1])

tier = next(v for k, v in sha3.items() if "sponge_tiered_kernelILi9E" in k)
bfly = [i for i, (_, t) in enumerate(tier) if "SHFL.BFLY" in t]
cands = [(s, e) for s, e in loops(tier) if s <= bfly[0] <= e]
s, e = min(cands, key=lambda se: se[1] - se[0])
dump(os.path.join(OUT, "keccak_pair_round.sass"), "sponge_tiered_kernel<9>, pair tier: loop body = four rounds of the split-lane permutation", tier[s:e + 1])
idx = [i for i, (_, t) in enumerate(tier) if "SHFL.IDX PT" in t]
dump(os.path.join(OUT, "keccak_warp_round.sass"), "sponge_tiered_kernel<9>, warp tier: first two rounds of the unrolled one-lane-per-thread permutation",
     tier[idx[0] - 6: idx[36] + 12])

# the step of the pair tier in front of the permutation: the loads of the next block as predicated LDGs on the straight
# line into the first round (round 2: they used to sit inside the absorb branch, and the first XOR of the permutation
# waited for them)
first_bfly = bfly[0]
ldg = [i for i, (_, t) in enumerate(tier) if "LDG.E.CONSTANT" in t and i < first_bfly]
dump(os.path.join(OUT, "pair_prefetch_before_permutation.sass"),
     "sponge_tiered_kernel<9>, pair tier: predicated loads of the next block, then the first instructions of the permutation",
     tier[max(0, ldg[-1] - 24): first_bfly + 4])

chain = next(v for k, v in sha3.items() if "sponge_chain_kernelILi17E" in k)
ns = [i for i, (_, t) in enumerate(chain) if "NANOSLEEP" in t]
at = [i for i, (_, t) in enumerate(chain) if t.split()[0].startswith(("ATOM", "RED")) or " ATOM" in t or " RED" in t]
if ns:
    dump(os.path.join(OUT, "chain_ticket_and_wait.sass"),
         "sponge_chain_kernel<17>: ticket (ATOM), job / block from the ticket, job 1 waiting for the job-0 block of its items",
         chain[max(0, at[0] - 6): ns[-1] + 10])
if len(at) > 1:
    dump(os.path.join(OUT, "chain_report.sass"), "sponge_chain_kernel<17>: a job-0 warp reports (fence, RED) after storing its states",
         chain[max(0, at[-1] - 40): at[-1] + 3])

vb = next(v for k, v in var.items() if "var_base_kernel" in k)
calls = collections.Counter(re.search(r"0x([0-9a-f]+)", t).group(1) for _, t in vb if t.startswith("CALL"))
rets = [i for i, (_, t) in enumerate(vb) if t.startswith("RET")]
for tgt, _ in calls.most_common():
    a0 = int(tgt, 16)
    i0 = next(i for i, (a, _) in enumerate(vb) if a == a0)
    i1 = next(r for r in rets if r >= i0)
    body = vb[i0:i1 + 1]
    wide = sum(1 for _, t in body if "IMAD.WIDE" in t)
    if wide > 150:
        dump(os.path.join(OUT, "fe_mul.sass"), f"fe_mul_call (ed448_var.cu): {len(body)} instructions, {wide} IMAD.WIDE", body)
    elif wide > 90:
        dump(os.path.join(OUT, "fe_sqr.sass"), f"fe_sqr_call (ed448_var.cu): {len(body)} instructions, {wide} IMAD.WIDE", body)
print(sorted(os.listdir(OUT)))
