#!/usr/bin/env python3
"""Static count of register-bank conflicts in the hot loops of a kernel, from `cuobjdump -sass` output.

    cuobjdump -sass bullet_envs_b200/csrc/libsnake_b200.so > /tmp/lib.sass
    python tools/sass_bank_conflicts.py /tmp/lib.sass snk_hyb_step_kernelILb1ELb0ELb0EE

For every backward-branch loop of 80..300 instructions with at least 40 fp32 multiplies it prints
(kind, instructions, conflicts, .reuse operands, fp instructions): kind = T/S (tensor-memory / shared-memory rows) + F/N (friction /
normal sweep, told apart by the MUFU of the cone projection).  A conflict = two source registers of one fp instruction in the same
bank (register number mod 4) and not served by the operand-reuse cache; on B200 each costs one issue cycle ("dispatch stall" in
ncu).  Used to screen operation-order variants of the solver without GPU time (profiles/README.md): the counts predicted the
measured ranking (17.7 -> 12.9 conflict cycles per contact and sweep = 4.50 -> 4.69 M env-steps/s)."""
import re, sys
def kernels(path):
    txt=open(path).read(); out={}
    for p in txt.split("Function : ")[1:]:
        out[p.split('\n')[0].strip()]=p
    return out
def ins_of(k):
    ins=[]
    for ln in k.split('\n'):
        m=re.match(r'\s+/\*([0-9a-f]{4,})\*/\s+(.*?);', ln)
        if m: ins.append((int(m.group(1),16), m.group(2)))
    return ins
def loops(ins):
    out=[]
    for i,(a,t) in enumerate(ins):
        if 'BRA' in t:
            m2=re.search(r'0x([0-9a-f]+)', t)
            if m2:
                tgt=int(m2.group(1),16)
                if tgt<a: out.append([x for x in ins if tgt<=x[0]<=a])
    return out
FP=('FFMA','FMUL','FADD','FMNMX','FSEL','MUFU.RSQ')
def metric(body):
    conf=0; reuse=0; nfp=0
    for a,t in body:
        tt=t.split()
        op=tt[0] if not t.startswith('@') else tt[1]
        if op not in FP: continue
        nfp+=1
        args=t[t.index(op)+len(op):].split(',')
        srcs=[]
        for s in args[1:]:
            m=re.match(r'\s*[-|!~]*\|?R(\d+)(\.reuse)?', s)
            if m:
                if m.group(2): reuse+=1
                else: srcs.append(int(m.group(1)))
        srcs=list(dict.fromkeys(srcs))
        conf+=len(srcs)-len(set(x%4 for x in srcs))
    return conf,reuse,nfp
def report(path, sub):
    for name,k in kernels(path).items():
        if sub not in name: continue
        res=[]
        for body in loops(ins_of(k)):
            n=len(body)
            if not (80<=n<=300): continue
            nfp=sum(1 for x in body if any(o in x[1] for o in ('FFMA','FMUL')))
            if nfp<40: continue
            kind='T' if any('LDTM' in x[1] for x in body) else 'S'
            mufu=sum('MUFU' in x[1] for x in body)
            if kind=='S' and not any('LDS' in x[1] for x in body): continue
            res.append((kind+('F' if mufu else 'N'),n)+metric(body))
        return res
if __name__=='__main__':
    for path,sub in [(a,b) for a,b in zip(sys.argv[1::2],sys.argv[2::2])]:
        print(path, report(path,sub))

def show(path, sub, kindwant):
    for name,k in kernels(path).items():
        if sub not in name: continue
        for body in loops(ins_of(k)):
            n=len(body)
            if n not in (130,131,103,104,94,96): continue
            kind='T' if any('LDTM' in x[1] for x in body) else 'S'
            mufu=sum('MUFU' in x[1] for x in body)
            if kind+('F' if mufu else 'N')!=kindwant: continue
            for a,t in body:
                tt=t.split(); op=tt[0] if not t.startswith('@') else tt[1]
                if op not in FP: continue
                args=t[t.index(op)+len(op):].split(',')
                srcs=[]
                for s in args[1:]:
                    m=re.match(r'\s*[-|!~]*\|?R(\d+)(\.reuse)?', s)
                    if m and not m.group(2): srcs.append(int(m.group(1)))
                srcs=list(dict.fromkeys(srcs))
                c=len(srcs)-len(set(x%4 for x in srcs))
                print(('**' if c else '  '), t, [x%4 for x in srcs])
            return
