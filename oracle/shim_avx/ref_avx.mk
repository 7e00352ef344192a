# oracle/shim_avx/ref_avx.mk — the reference's OWN sources built like `make -C oracle ref` (oracle/Makefile: same flags,
# same stand-in headers), with the stand-in's dynamic-size sums on 8-float AVX packets (packet8_sum.h, forced
# include): the reference as built against an Eigen that vectorises with AVX.  Test infrastructure, NOT the product.
#
#   make -C oracle -f shim_avx/ref_avx.mk REF=<reference checkout>   ->  oracle/_ref_avx/libictrack_ref.so
include Makefile
.DEFAULT_GOAL := ref_avx

ref_avx: _ref_avx/libictrack_ref.so
_ref_avx/libictrack_ref.so: ref_capi.cpp $(REFSRC) shim/Eigen/Core shim_avx/packet8_sum.h shim/opencv2/core/core.hpp
	mkdir -p _ref_avx
	$(CXX) $(CXXFLAGS) -include shim_avx/packet8_sum.h -shared -o $@ ref_capi.cpp $(REFSRC)
clean_ref_avx:
	rm -rf _ref_avx
.PHONY: ref_avx clean_ref_avx
