#!/bin/bash
# SASS mnemonics that show which hardware paths the kernels use (B200_PROFILING.md "What proves a
# Blackwell-native kernel"): counts per object file of libmmb_b200.so.  Runs on the CPU box (no GPU needed).
cd "$(dirname "$0")/../multimodal-baselines_b200" || exit 1
python build.py > /dev/null
for f in gram_tc sif_embed remove_pc peer_comm pc_solve mmb_step; do
  echo "== csrc/$f.cu"
  cuobjdump -sass build/$f.o 2>/dev/null | grep -oE "\b(UTC[A-Z]*MMA[.A-Z0-9_]*|UTMALDG[.A-Z0-9_]*|UTMAPF[.A-Z0-9_]*|UTCBAR[.A-Z0-9_]*|UTCATOMSWS[.A-Z0-9_]*|LDTM[.A-Z0-9_x]*|STTM[.A-Z0-9_x]*|SYNCS[.A-Z0-9_]*|FFMA2|MATCH\.ANY|LDG\.E\.NA\.128[.A-Z]*|LDG\.E\.128[.A-Z]*|DFMA|ACQBULK|HMMA[.A-Z0-9_]*|ATOMG[.A-Z0-9_]*|LD\.E\.[A-Z0-9.]*SYS[.A-Z0-9]*|ST\.E\.[A-Z0-9.]*SYS[.A-Z0-9]*)" | sort | uniq -c | sort -rn
done
echo "== csrc/gram_tc.cu: A-operand collector flags on the tcgen05 MMAs (operand suffixes, not part of the mnemonic)"
cuobjdump -sass build/gram_tc.o 2>/dev/null | grep -oE "UTCHMMA gdesc\[UR[0-9]+\](\.A_REUSE)?(\.A_KEEP)?" | sed -E 's/\[UR[0-9]+\]/[..]/' | sort | uniq -c | sort -rn
