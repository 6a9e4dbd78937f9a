"""Analysis script (not a test; uses the CPU oracle, so it lives under tests/): how much of an EARLY block's outcome depends on the
~95 table updates inside the block?  Block 0 of the bench stream is run twice through the oracle -- (A) with the reference's sync
schedule, (B) as ONE segment with a single sync at the end -- and the per-base records and the push rows are compared.

Result (round 1, block 0, 51 000 reads, -gs 100):
    p pushes 13668000 vs 13667948 (same distinct set), s pushes 6681000 identical sequence, b pushes 6477000 identical sequence
    records 7038000: counts differ 0.945 %, level differ 0.943 %, cor_pos differ 0 %
      level none 96.45 % of the records, none differ | level pmer 0.94 %, ALL differ | smer 0.27 %, 0.037 % differ | bmer 2.33 %, 0.079 % differ
i.e. the trajectory (registers, repairs, s-/b-mer pushes) of an early block does not depend on the intra-block syncs at all; what does
is the p-mer level (the 2-bit array has no thread-local twin, so only a sync makes a p-mer visible) and a handful of s-/b-level counts.
This is the evidence behind DESIGN.md's round-2 plan (block-level pass + versioned fix-up).   Run: python tests/probe_block_visibility.py (~6 min)"""
import os, sys, time, numpy as np
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from fqsqueezer_b200 import synth, schedule as S, engine as E
from oracle import oracle as O
import bench
G=bench.GENOME; genome=synth.make_genome(G, bench.SEED)
pref,p,s,b=E.kmer_params(100)
def run(g, per_segment):
    o=O.OracleEngine(p,s,b,pref)
    codes=bench.block_codes(genome,g)
    slab,off,ln=bench.codes_to_slab(codes)
    n=len(off)
    ns=S.calc_no_synchronizations(g,n,1) if per_segment else 0
    o.block_start()
    rows=[[],[],[]]; recs=[]
    for a,bb in S.segments(0,n,ns):
        r,d=o.segment(slab,off[a:bb],ln[a:bb]); recs.append(r)
        for w in range(3): rows[w].append(o.pending(w, 1<<25))
        o.sync()
    o.close()
    return np.concatenate(recs), [np.concatenate(x) for x in rows]
ra,A=run(0,True); rb,B=run(0,False)
for w,nm in enumerate('psb'):
    a,b_=A[w],B[w]
    same_len=len(a)==len(b_)
    print(nm,'pushes',len(a),len(b_),'identical sequence' if same_len and np.array_equal(a,b_) else 'differ')
    if not(same_len and np.array_equal(a,b_)):
        ua,ca=np.unique(a,return_counts=True); ub,cb=np.unique(b_,return_counts=True)
        only_a=np.setdiff1d(ua,ub).size; only_b=np.setdiff1d(ub,ua).size
        print('   distinct',ua.size,ub.size,'only in A',only_a,'only in B',only_b)
a=ra[ra['pos']<0xFFFFFFF0]; bb=rb[rb['pos']<0xFFFFFFF0]
d_counts=(a['c']!=bb['c']).any(axis=1); d_lev=a['level']!=bb['level']; d_cor=a['cor_pos']!=bb['cor_pos']
print('records',len(a),'counts differ %.3f%% level differ %.3f%% cor_pos differ %.4f%%'%(100*d_counts.mean(),100*d_lev.mean(),100*d_cor.mean()))
for lv in range(6):
    m=(a['level']==lv)
    if m.any(): print('  level',lv,'share %.2f%%'%(100*m.mean()),'differ within %.3f%%'%(100*(d_counts|d_lev)[m].mean()))
