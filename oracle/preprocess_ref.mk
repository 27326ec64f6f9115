# TEST INFRASTRUCTURE ONLY. Builds _ref/libpreprocess_ref.so: the REFERENCE's own src/preprocess.cpp compiled
# unmodified, in place, from $(REF), next to preprocess_ref_wrap.cpp (only when $(REF) exists; the built .so travels
# with the working tree; no reference source is copied into this repo).  preprocess.h includes "common_lib.h", which
# resolves to the stand-in in shim/preprocess/ because $(REF)/include is deliberately not on the include path.
#     make -C oracle -f preprocess_ref.mk
REF ?= /root/reference
CXX = g++
# the reference's own optimisation level (CMakeLists.txt:9 "-O3", no -march) + OpenMP (omp_get_wtime)
CXXFLAGS_REF = -O3 -std=c++17 -fPIC -fopenmp -w

all:
	@if [ -f $(REF)/src/preprocess.cpp ]; then \
	  mkdir -p _ref && \
	  echo "building _ref/libpreprocess_ref.so from $(REF)/src/preprocess.cpp" && \
	  $(CXX) $(CXXFLAGS_REF) -shared -Ishim/preprocess -I$(REF)/src -o _ref/libpreprocess_ref.so \
	      preprocess_ref_wrap.cpp $(REF)/src/preprocess.cpp ; \
	else echo "reference tree not present at $(REF): keeping prebuilt _ref/libpreprocess_ref.so (if any)"; fi

clean:
	rm -f _ref/libpreprocess_ref.so
.PHONY: all clean
