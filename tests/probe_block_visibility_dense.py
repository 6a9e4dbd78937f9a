"""Analysis script (not a test; uses the CPU oracle): companion of probe_block_visibility.py for POPULATED tables, in a regime ten
times denser than BASELINE config 2 (10 Mbp genome: three prior blocks = 2.3x coverage in the tables, the probed block adds 0.77x of
its own, where config 2 adds 0.077x per block).  The probed block is run (A) with the reference's 96 syncs and (B) as one segment.

Result (round 1):
    p pushes 9701408 vs 10648448 (B pushes more: pmer_insert is suppressed less often when counts are seen later), s pushes 6681000 both
    (26 123 of 5.16 M distinct only in B), b pushes 6481522 vs 6479983 (30 933 of 5.08 M distinct only in B)
    records 7038000: counts differ 20.5 %, level 1.05 %, cor_pos 1.25 %; reads with any differing record 54 %
      level none 10.9 % (0.2 % differ) | pmer 10.0 % (23 %) | smer 5.3 % (18 %) | bmer 73.9 % (24 %)
i.e. with populated tables the cross-segment dependence is carried by COUNT VALUES (a b-mer seen once more), rarely by the trajectory
(cor_pos 1.25 %, pushes 0.5 %) -- at ten times the real density.  At config-2 density expect about a tenth of it: the versioned
counts of DESIGN.md's round-2 plan are needed for ~2 % of the records of a late early block, the re-walk set stays small."""
import os, sys, time, numpy as np
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from fqsqueezer_b200 import synth, schedule as S, engine as E
from oracle import oracle as O
import bench
G=10_000_000; genome=synth.make_genome(G, 5)
pref,p,s,b=E.kmer_params(100)
PRIOR=3
def run(per_segment_last):
    o=O.OracleEngine(p,s,b,pref)
    for g in range(PRIOR+1):
        codes,_=synth.make_reads(genome, bench.READS_PER_BLOCK, L=bench.L, seed=100+g)
        slab,off,ln=bench.codes_to_slab(codes)
        n=len(off)
        last = g==PRIOR
        ns=S.calc_no_synchronizations(g,n,1) if (not last or per_segment_last) else 0
        o.block_start()
        rows=[[],[],[]]; recs=[]
        for a,bb in S.segments(0,n,ns):
            r,d=o.segment(slab,off[a:bb],ln[a:bb])
            if last:
                recs.append(r)
                for w in range(3): rows[w].append(o.pending(w, 1<<25))
            o.sync()
    o.close()
    return np.concatenate(recs), [np.concatenate(x) for x in rows]
ra,A=run(True); rb,B=run(False)
for w,nm in enumerate('psb'):
    a,b_=A[w],B[w]
    if len(a)==len(b_) and np.array_equal(a,b_): print(nm,'pushes',len(a),'identical sequence')
    else:
        ua=np.unique(a); ub=np.unique(b_)
        print(nm,'pushes',len(a),len(b_),'distinct',ua.size,ub.size,'only in A',np.setdiff1d(ua,ub).size,'only in B',np.setdiff1d(ub,ua).size)
a=ra[ra['pos']<0xFFFFFFF0]; bb=rb[rb['pos']<0xFFFFFFF0]
print('records',len(a),len(bb))
if len(a)==len(bb):
    d_counts=(a['c']!=bb['c']).any(axis=1); d_lev=a['level']!=bb['level']; d_cor=a['cor_pos']!=bb['cor_pos']
    print('counts differ %.3f%% level differ %.3f%% cor_pos differ %.4f%%'%(100*d_counts.mean(),100*d_lev.mean(),100*d_cor.mean()))
    for lv in range(6):
        m=(a['level']==lv)
        if m.any(): print('  level',lv,'share %.2f%%'%(100*m.mean()),'differ within %.3f%%'%(100*(d_counts|d_lev|d_cor)[m].mean()))
    starts=np.flatnonzero(a['pos']==pref)
    anyd=np.add.reduceat((d_counts|d_lev|d_cor).astype(np.int64),starts)>0
    print('reads with any differing record %.2f%%'%(100*anyd.mean()))
