#!/bin/bash
# SASS evidence for the hot kernels of libdnagpu.so: opcode histogram + the memory instructions of each.
#   tools/sass_excerpt.sh > profiles/r02_sass_hot_kernels.txt
SO=dna-sequences-pg-extension_b200/libdnagpu.so
echo "# cuobjdump -sass of $SO (sm_100a), $(date -u +%F); nvcc $(nvcc --version | grep release | sed 's/.*release //')"
for pat in 'k_extract4ILi0' 'k_part_scatter_seqILi0ELb0E' 'k_part_scatter_keysILb0ELi32' 'k_count_buckets_bins' \
           'k_collect_ownedILi4ELi3ELb0' 'k_collect_ownedILi4ELi0ELb0' 'k_filter_saILi1' 'k_filter_collectILi1'; do
  fn=$(cuobjdump -sass $SO 2>/dev/null | grep "Function :" | grep "$pat" | head -1 | sed 's/.*Function : //')
  [ -z "$fn" ] && continue
  echo
  echo "## $fn"
  body=$(cuobjdump -sass -fun "$fn" $SO 2>/dev/null | grep -E "^\s+/\*[0-9a-f]{4}\*/")
  echo "instructions: $(echo "$body" | wc -l)"
  echo "opcode histogram (top 16):"
  echo "$body" | awk '{print $2}' | sed 's/\..*//;s/;//' | grep -v '^@' | sort | uniq -c | sort -rn | head -16 | awk '{printf "  %6d %s\n",$1,$2}'
  echo "global / shared memory instructions (distinct forms):"
  echo "$body" | grep -oE "(LDG|STG|LDS|STS|ATOMS|ATOMG|RED|LDSM|UBLKCP|LDGSTS)[A-Z0-9_.]*" | sort | uniq -c | sort -rn | awk '{printf "  %6d %s\n",$1,$2}'
done
