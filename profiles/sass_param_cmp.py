"""SASS of every kernel of a parent hz_mcts.cu cubin against this tree's: identical, identical apart from the parameter
constant-bank offsets (c[0x0][...]), or different.  Kernels are matched by name, with the mode-off template arguments
that round 10 appended (GUMBEL = false, the hz_gumbel_args parameter) filled in.
Usage: python profiles/sass_param_cmp.py parent.cubin new.cubin   (cubins from nvcc -cubin with build.py's flags)
"""
import subprocess,re,sys
def funcs(cubin):
    out=subprocess.run(["cuobjdump","-sass",cubin],capture_output=True,text=True).stdout
    fs={}
    cur=None
    for line in out.splitlines():
        m=re.match(r"\s+Function : (\S+)",line)
        if m: cur=m.group(1); fs[cur]=[]; continue
        if cur and re.match(r"\s+/\*[0-9a-f]{4}\*/",line):
            ins=line.split(";")[0]
            ins=re.sub(r"/\*[0-9a-f]+\*/","",ins).strip()
            fs[cur].append(ins)
    return fs
P=funcs(sys.argv[1]); N=funcs(sys.argv[2])
def newname(p):
    if 'k_tree_select' in p:
        return p.replace("EEEv7hz_tree","ELb0EEEv7hz_tree").replace("EvalCacheArgs","EvalCacheArgs14hz_gumbel_args")
    if 'k_tree_expand_backup' in p:
        return p.replace("EEEv7hz_treePKfS3_iS3_d","ELb0EEEv7hz_treePKfS3_iS3_dPf")
    return p
same=offs=diff=0
for p,ins in P.items():
    n=newname(p)
    if n not in N: print("MISSING",p,n); diff+=1; continue
    a,b=ins,N[n]
    if a==b: same+=1; continue
    norm=lambda L:[re.sub(r"c\[0x0\]\[0x[0-9a-f]+\]","c[0x0][X]",x) for x in L]
    if norm(a)==norm(b): offs+=1
    else:
        diff+=1; print("DIFF",p,len(a),len(b))
print(f"{len(P)} parent kernels: {same} identical, {offs} identical apart from constant-bank offsets, {diff} different")
