#!/bin/bash
# Blackwell-native evidence from the shipped library: SASS mnemonic counts + excerpts (run on the CPU box).
SO=hipporag_b200/libhrag_b200.so
OUT=profiles/r2_sass_evidence.txt
{
  echo "# cuobjdump -sass $SO  (sm_100a), $(date -u +%Y-%m-%d)"
  echo "## mnemonic counts over the whole library"
  cuobjdump -sass $SO 2>/dev/null | grep -oE "\b(UTCHMMA(\.2CTA)?|UTMALDG\.2D(\.GATHER4)?|UTMALDG\.[A-Z0-9.]+|LDTM\.[x0-9A-Za-z.]+|UTCBAR[A-Z0-9.]*|UBLKCP[A-Z0-9.]*|UTMAPF[A-Z0-9.]*|SYNCS[A-Z0-9.]*|HMMA[A-Z0-9.]*|LDG\.E\.128\.CONSTANT|LDG\.E\.NA\.128\.CONSTANT|RED\.[A-Z0-9.]+|ATOMG[A-Z0-9.]*)" | sort | uniq -c | sort -rn
  for fn in k_sim_tcILb1ELi1E k_sim_tcILb1ELi2E k_sweep_hILb1ELi0ELb0EE; do
    echo; echo "## excerpt: $fn"
    cuobjdump -sass $SO 2>/dev/null | awk -v f="$fn" '$0 ~ "Function : " && $0 ~ f {p=1} p{print} p && /EXIT/{c++} c>=1 && p{if (++n>400) exit}' \
      | grep -E "Function :|UTCHMMA|UTMALDG|LDTM|UTCBAR|UBLKCP|SYNCS|LDG\.E|STG\.E|HADD2|FFMA|ATOMG|RED\.|MEMBAR|ST\.E.*SYS|LD\.E.*SYS|BAR\.SYNC" | cut -c1-120 | head -60
  done
} > $OUT
wc -l $OUT
