#!/usr/bin/env python3
"""SASS opcode histogram of the network kernels: python tools/sass_opcodes.py > profiles/r02_net_sass_opcodes.txt
(cuobjdump -sass of the sm_100a object; proves which kernels issue tcgen05.mma (UTC*MMA), tcgen05.ld/st (LDTM/STTM), bulk copies
(UBLKCP), tcgen05.commit (UTCBAR) and that none falls back to mma.sync (HMMA))."""
import collections
import re
import subprocess
import sys

OBJ = sys.argv[1] if len(sys.argv) > 1 else "onitama_alphazero_b200/csrc/onb_net.o"
COLS = ["UTCHMMA", "UTCHMMA.2CTA", "UTCQMMA", "UTCBAR", "UTCATOMSWS", "LDTM", "STTM", "UBLKCP", "SYNCS", "HMMA", "STS", "LDS", "LDG", "STG", "FFMA", "F2FP"]
out = subprocess.run(["cuobjdump", "-sass", OBJ], capture_output=True, text=True, check=True).stdout
names = subprocess.run(["cu++filt"], input="\n".join(re.findall(r"Function : (\S+)", out)), capture_output=True, text=True).stdout.split("\n")
hist, order, cur, i = {}, [], None, 0
for line in out.split("\n"):
    m = re.search(r"Function : (\S+)", line)
    if m:
        d = names[i]
        i += 1
        d = re.sub(r"^void ", "", d)
        d = re.sub(r"onb::\(anonymous namespace\)::|onb::<unnamed>::", "", d)
        d = re.sub(r"\((int|bool)\)", "", d)  # template arguments print as (int)2, (bool)1
        cur = re.sub(r"\(.*", "", d)
        hist[cur] = collections.Counter()
        order.append(cur)
        continue
    m = re.match(r"\s+/\*[0-9a-f]{4,}\*/\s+(?:@!?U?P\d+\s+)?([A-Z0-9_]+)", line)
    if m and cur:
        op = m.group(1)
        hist[cur][op] += 1
        hist[cur]["total"] += 1
        if "UTCHMMA.2CTA" in line:  # tcgen05.mma.cta_group::2 (counted in UTCHMMA as well)
            hist[cur]["UTCHMMA.2CTA"] += 1
print("# SASS opcode histogram of the network kernels (python tools/sass_opcodes.py: cuobjdump -sass %s, sm_100a)" % OBJ)
print("# tcgen05.mma -> UTC*MMA, tcgen05.ld/st -> LDTM/STTM, cp.async.bulk -> UBLKCP, tcgen05.commit -> UTCBAR, tcgen05.alloc -> UTCATOMSWS,")
print("# mbarrier -> SYNCS. Shipped: k_net_forward_x3p<true> (ONB_NET_F32: CTA pairs, tcgen05 cta_group::2), k_net_forward_x3p<false> (its")
print("# single-CTA fallback), k_net_forward_f16q<true|false> (ONB_NET_F16), k_net_forward<false, false> (ONB_NET_TF32); the others are plain builds")
print()
print("%-44s" % "kernel" + "".join("%13s" % c for c in COLS) + "%9s" % "total")
for k in order:
    if "k_net_forward" in k:
        print("%-44s" % k + "".join("%13d" % hist[k][c] for c in COLS) + "%9d" % hist[k]["total"])
