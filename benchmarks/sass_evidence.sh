#!/usr/bin/env bash
# Counts the SASS mnemonics that prove which hardware paths the built objects use (B200_PROFILING.md): tcgen05
# (UTCHMMA, LDTM, UTCBAR, UTCATOMSWS = tcgen05.alloc), TMA (UTMALDG), mbarrier (SYNCS.*), system-scope
# peer loads/stores (LDG/STG ...STRONG.SYS), 128-bit streaming loads, dp4a.  Runs on the CPU build host:
#   python -m cor_b200.build && benchmarks/sass_evidence.sh > profiles/rNN_sass_evidence.txt
cd "$(dirname "$0")/.." || exit 1
for o in pool_umma sim_umma sim_umma_ts nce_bwd_umma gemm_umma pool_bwd_umma peer mask_prep pool_stream sim_stream seg_loss seg_strip dwconv ln_rows ew; do
  echo "== cor_b200/build/$o.o"
  cuobjdump -sass "cor_b200/build/$o.o" 2>/dev/null |
    grep -oE "\b(UTCHMMA|UTCHMMA[.A-Z0-9_]*|FFMA2|FADD2|FMNMX3|STTM[.A-Za-z0-9_]*|UTMAPF[.A-Z0-9_]*|UTMALDG[.A-Z0-9_]*|UTCBAR[.A-Z0-9_]*|LDTM[.A-Za-z0-9_]*|UTCATOMSWS[.A-Z0-9_]*|SYNCS[.A-Z0-9_]*|LDG\.E\.128[.A-Z0-9_]*|LDG\.E\.[A-Z0-9_.]*SYS[.A-Z0-9_]*|STG\.E\.[A-Z0-9_.]*SYS[.A-Z0-9_]*|MEMBAR[.A-Z0-9_]*|IDP\.4A[.A-Z0-9_]*|MUFU\.EX2|REDUX[.A-Z0-9_]*)" |
    sort | uniq -c | sort -rn | head -14
done
