#!/usr/bin/env python
"""Offline replay of the association's work distribution on C1 data (CPU only, oracle + NumPy): per query the points in its
own 0.5 m cell, in the 27-cell cube, and in the cells that survive the bound of the own cell / the final bound; and how
well 32 consecutive queries balance under different orderings (Morton, own-cell population, exact work).  The numbers
quoted in DESIGN.md §5 come from here.

    python tools/assoc_work_analysis.py
"""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, oracle
from liodom_b200 import synth
scans,gt = synth.sequence("hdl64",1000,18)
op = oracle.make_params(prev_frames=15)
odo = oracle.Odometer(op)
edges=[oracle.extract_scan(op,s)[0] for s in scans]
for f in range(17): pose,_=odo.process(edges[f])
win,_=odo.window(); W=win[:,:3]
o,pv=odo.get_pose()
pred = o @ (np.linalg.inv(pv) @ o)
q = (edges[17][:,:3].astype(np.float64) @ pred[:3,:3].T + pred[:3,3]).astype(np.float32)
cell=0.5
wc = np.floor(W/cell).astype(np.int64); qc=np.floor(q/cell).astype(np.int64)
from collections import defaultdict
key=lambda c: (c[:,0]+5000)*100000000+(c[:,1]+5000)*10000+(c[:,2]+5000)
wk=key(wc); uk,inv,cnt=np.unique(wk,return_inverse=True,return_counts=True)
d=dict(zip(uk.tolist(),cnt.tolist()))
print("map pts",len(W),"cells",len(uk),"mean pts/cell",cnt.mean(),"max",cnt.max(), "pcts",np.percentile(cnt,[50,90,99]))
# per query counts
order=np.argsort(wk); 
import itertools
offs=[(a,b,c) for a in (-1,0,1) for b in (-1,0,1) for c in (-1,0,1)]
n_own=np.zeros(len(q),int); n27=np.zeros(len(q),int); ncell27=np.zeros(len(q),int)
# exact 5th best distance via brute force per query among 27 cells
bucket=defaultdict(list)
for i,k in enumerate(wk.tolist()): bucket[k].append(i)
npr=np.zeros(len(q),int); ncellpr=np.zeros(len(q),int)
for i in range(len(q)):
    c=qc[i]; cand=[]
    k0=int((c[0]+5000)*100000000+(c[1]+5000)*10000+(c[2]+5000))
    n_own[i]=d.get(k0,0)
    segs=[]
    for a,b,cc in offs:
        kk=int((c[0]+a+5000)*100000000+(c[1]+b+5000)*10000+(c[2]+cc+5000))
        n=d.get(kk,0)
        if n: ncell27[i]+=1; n27[i]+=n; segs.append((a,b,cc,kk,n))
    allc=np.concatenate([bucket[s[3]] for s in segs]) if segs else np.zeros(0,int)
    if len(allc)>=5:
        d2=((W[allc]-q[i])**2).sum(1); k5=np.sort(d2)[4]
    else: k5=1.0
    k5=min(k5,1.0)
    for a,b,cc,kk,n in segs:
        lo=(c+np.array([a,b,cc]))*cell; hi=lo+cell
        g=np.maximum(0,np.maximum(lo-q[i],q[i]-hi)); dm=(g**2).sum()
        if dm<=k5: npr[i]+=n; ncellpr[i]+=1
print("per query: own mean %.1f, 27-cell mean %.1f (cells %.1f), with final-bound pruning mean %.1f (cells %.1f)"%(n_own.mean(),n27.mean(),ncell27.mean(),npr.mean(),ncellpr.mean()))
print("pruned pcts", np.percentile(npr,[10,50,90,99,100]))
# morton order
def spread(v):
    v=v&0x3ff; v=(v|(v<<16))&0x030000ff; v=(v|(v<<8))&0x0300f00f; v=(v|(v<<4))&0x030c30c3; v=(v|(v<<2))&0x09249249; return v
mk=spread(qc[:,0].astype(np.uint32))|(spread(qc[:,1].astype(np.uint32))<<1)|(spread(qc[:,2].astype(np.uint32))<<2)
mo=np.argsort(mk,kind='stable')
for name,arr in (("pruned",npr),("all27",n27),("own",n_own)):
    a=arr[mo]; nw=len(a)//32
    a=a[:nw*32].reshape(nw,32)
    print(name,"warp efficiency mean/max = %.3f ; sum(max)*32 / sum = %.2f"%((a.mean(1)/np.maximum(a.max(1),1)).mean(), a.max(1).sum()*32/a.sum()))
    a4=np.ceil(arr[mo][:nw*32].reshape(nw,32)/4)
    print("   iterations of 4: warp max sum", a4.max(1).sum(), "ideal", a4.sum()/32)
# sorted by work
a=np.sort(npr)[:len(npr)//32*32].reshape(-1,32)
print("if sorted by work: eff", a.sum()/(a.max(1).sum()*32))
print("---- proxies")
def eff(order, arr):
    a=arr[order]; nw=len(a)//32; a=a[:nw*32].reshape(nw,32); return a.sum()/(a.max(1).sum()*32)
for name,proxy in (("n_own",n_own),("n27",n27),("ncell27",ncell27)):
    o=np.argsort(proxy,kind='stable')
    print(name,"sorted: eff on pruned work %.3f ; corr %.3f"%(eff(o,npr), np.corrcoef(proxy,npr)[0,1]))
print("morton eff", eff(mo,npr))
# what if bound came from own cell only (5th best within own cell) -> work = cells with dmin<=k5own
npr2=np.zeros(len(q),int)
for i in range(len(q)):
    c=qc[i]
    k0=int((c[0]+5000)*100000000+(c[1]+5000)*10000+(c[2]+5000))
    own=bucket.get(k0,[])
    if len(own)>=5:
        d2=((W[own]-q[i])**2).sum(1); k5=min(np.sort(d2)[4],1.0)
    else: k5=1.0
    tot=0
    for a,b,cc in offs:
        kk=int((c[0]+a+5000)*100000000+(c[1]+b+5000)*10000+(c[2]+cc+5000))
        n=d.get(kk,0)
        if not n: continue
        lo=(c+np.array([a,b,cc]))*cell; hi=lo+cell
        g=np.maximum(0,np.maximum(lo-q[i],q[i]-hi)); dm=(g**2).sum()
        if dm<=k5: tot+=n
    npr2[i]=tot
print("own-bound pruning: mean cands %.1f ; eff if sorted by it: %.3f, morton %.3f"%(npr2.mean(), eff(np.argsort(npr2),npr2), eff(mo,npr2)))
print("frac queries with own>=5:", (n_own>=5).mean())
