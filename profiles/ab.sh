# A/B of library builds, two rounds: LIBS = paths of other builds of the library (CAMCAL_B200_LIB, e.g. the parent
# commit's) and "default" = the built library, in the order they alternate; WL/CO = workload / coords
for r in 1 2; do for so in ${LIBS:?"LIBS: library paths and/or default"}; do
  if [ "$so" = default ]; then python profiles/ktime.py ${WL:-c2} ${CO:-f64} 2>&1 | tail -1
  else CAMCAL_B200_LIB=$(realpath "$so") python profiles/ktime.py ${WL:-c2} ${CO:-f64} 2>&1 | tail -1; fi
done; done
