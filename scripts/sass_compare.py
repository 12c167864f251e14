"""Per-subroutine SASS comparison of two builds of the solve kernel (no GPU needed): the noinline device functions keep
their own labels inside the kernel's section, so a change that should not touch a hot function can be checked by
comparing that function's instruction stream.

    cuobjdump -xelf all old.o; nvdisasm -c *.cubin > old.txt      (same for new.o -> new.txt)
    python scripts/sass_compare.py old.txt new.txt

Used in round 1 after an unused call site in qp_solve_gi had cost 5 % (see DESIGN.md): ptxas re-rolls MOV / IMAD.MOV
encodings between builds, so equal length + same opcode classes is the practical criterion: such functions are listed
as REROLL and not counted as differing."""
import re, collections, sys
def parse(path):
    # key: (kernel variant, mangled function name after the unit-specific namespace prefix), i.e. the name together
    # with its template arguments and parameter types, so that the instantiations of one template stay apart
    res = collections.OrderedDict(); cur=None
    for line in open(path):
        m = re.match(r'^(\$?\S+):\s*$', line)
        if m and ('dgsqp_solve_kernel' in m.group(1)) and not m.group(1).startswith('.L'):
            name = m.group(1)
            # kernel variant + internal function name
            var = 'T' if 'kernelILb1' in name.split('$')[1 if name.startswith('$') else 0] else 'F'
            mm = re.search(r'\$_ZN\d+_INTERNAL_\w+?_GLOBAL__N__\w+?_cu_[0-9a-f]{8}(\d+\w+)', name)
            cur = (var, mm.group(1) if mm else 'ENTRY'); res[cur]=[]; continue
        m = re.match(r'\s*/\*[0-9a-f]{4,}\*/\s+(.*?);', line)
        if m and cur is not None:
            ins = re.sub(r'0x[0-9a-f]+','IMM', m.group(1)); ins = re.sub(r'`\([^)]*\)','LBL',ins)
            res[cur].append(ins)
    return res
def short(fn):
    m = re.match(r'(\d+)', fn)
    return fn if not m else fn[len(m.group(1)):len(m.group(1)) + int(m.group(1))] + ' ' + fn[len(m.group(1)) + int(m.group(1)):]
# integer moves / adds / shifts that ptxas re-chooses among (ALU vs FMA pipe) when register allocation shifts
INT = {'MOV', 'IMAD.MOV', 'IMAD.MOV.U32', 'HFMA2', 'IADD3', 'IADD3.X', 'VIADD', 'IMAD', 'IMAD.IADD', 'IMAD.X', 'IMAD.U32',
       'IMAD.SHL.U32', 'SHF.L.U32', 'LEA'}
def opclasses(ins):
    ops = [i.split()[1] if i.startswith('@') else i.split()[0] for i in ins]
    return collections.Counter('INT' if o in INT else o for o in ops)
A = parse(sys.argv[1]); B = parse(sys.argv[2])
print(len(A), len(B))
tot = rer = 0
for k in B:
    v,f = k
    if v!='T': continue
    a = A.get(k)
    if a is None: print('NEW', v, short(f), len(B[k])); continue
    if a == B[k]: continue
    if len(a) == len(B[k]) and opclasses(a) == opclasses(B[k]):
        print('REROLL', v, short(f), len(a)); rer += 1      # same length, same opcodes up to integer re-rolls
    else:
        ca, cb = opclasses(a), opclasses(B[k])
        d = {o: cb[o] - ca[o] for o in set(ca) | set(cb) if cb[o] != ca[o]}
        print('DIFF', v, short(f), len(a), len(B[k]), d); tot += 1
print('differing SM=true functions:', tot, 'of', sum(1 for k in B if k[0]=='T'), '(plus', rer, 'with integer re-rolls only)')
