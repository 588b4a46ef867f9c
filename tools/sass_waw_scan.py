#!/usr/bin/env python
"""Scan a kernel's SASS for a LOAD DESTINATION OVERWRITTEN BEFORE IT IS READ within the next 14 straight-line instructions:
the write has to wait for the load (write-after-write on the scoreboard), i.e. the warp stalls on a prefetch it has just
issued.  Found this way: pass A's 128-bit table-entry load whose dead third word ptxas reused for a flag byte (12.6 % of all
stall samples on one PRMT, DESIGN.md 7).  Predicated select patterns (load a default, overwrite it under a predicate) show up
too and are harmless when the load is a shared-memory one.
usage: python tools/sass_waw_scan.py openkitchen_b200/lib/libopenkitchen_b200.so beam_step_kernelILb1ELb0E"""
import re,subprocess,sys
lib=sys.argv[1]; pat=sys.argv[2]
out=subprocess.run(["cuobjdump","-sass",lib],capture_output=True,text=True).stdout
funcs={}; cur=None
for line in out.splitlines():
    m=re.search(r"Function : (\S+)",line)
    if m: cur=m.group(1); funcs[cur]=[]; continue
    m=re.match(r"\s+/\*([0-9a-f]+)\*/\s+(.*?);",line)
    if m and cur: funcs[cur].append((int(m.group(1),16),m.group(2).strip()))
width={"128":4,"64":2}
def regs(tok):
    return [int(x) for x in re.findall(r"\bR(\d+)\b",tok)]
for f,ins in funcs.items():
    if pat not in f: continue
    print("==",f,len(ins))
    for i,(a,t) in enumerate(ins):
        m=re.match(r"(@!?U?P\d+\s+)?(LDG|LDS|LDL|LD|LDC|ATOMS|ATOMG|SHFL|I2F|F2I|MUFU|DMUL|DFMA|DADD|F2F|I2FP)\S*\s+(?:P\w+,\s*)?R(\d+)",t)
        if not m: continue
        op=m.group(2)
        if op not in("LDG","LDS","LDL","LD","ATOMS","ATOMG"): continue
        w=1
        mm=re.search(r"\.(128|64)\b",t.split()[0] if not t.startswith('@') else t.split()[1])
        if mm: w=width[mm.group(1)]
        d0=int(m.group(3)); dests=set(range(d0,d0+w))
        # scan forward up to 12 instrs in straight line
        for j in range(i+1,min(i+14,len(ins))):
            tj=ins[j][1]
            if re.match(r"(@!?U?P\d+\s+)?(BRA|BSYNC|EXIT|CALL|RET|BAR|WARPSYNC|JMP)",tj): break
            parts=tj.split(None,1)
            body=tj
            # dest = first R after opcode
            mj=re.match(r"(@!?U?P\d+\s+)?(\S+)\s+(.*)",tj)
            if not mj: continue
            ops=mj.group(3).split(",")
            dst=regs(ops[0]) if not mj.group(2).startswith(("ST","RED","BAR")) else []
            src=set(regs(",".join(ops[1:]))) if dst else set(regs(mj.group(3)))
            # 64-bit sources approx ignored
            if src & dests: break
            if dst and dst[0] in dests:
                print(f"  {a:05x} {t[:60]:60s} -> {ins[j][0]:05x} {tj[:50]}")
                break
