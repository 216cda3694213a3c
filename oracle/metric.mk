# oracle/metric.mk -- the checkers of the spatial metric (manhattan_spatial_dist).  TEST INFRASTRUCTURE ONLY.
#
#   liboracle_metric.so          : oracle/spatial_metric.c (the plain-C restatement, which includes slic_oracle.c)
#   _ref/libfslic_ref_metric.so  : oracle/ref_shim_metric.cpp against the UNMODIFIED reference objects of
#                                  _ref/libfslic_ref.so (oracle/Makefile); only built where $(REF) exists.
#
#   make -C oracle -f metric.mk liboracle_metric.so ref
REF ?= /root/reference
CXX = /usr/bin/g++
CC  = /usr/bin/gcc
REF_FLAGS = -std=c++11 -O3 -fopenmp -fPIC -DUSE_AVX2 -mavx2 -mfma -w

all: liboracle_metric.so ref

liboracle_metric.so: spatial_metric.c slic_oracle.c
	$(CC) -O2 -fPIC -std=c99 -shared spatial_metric.c -o liboracle_metric.so -lm

ref:
	@if [ -d $(REF)/src ]; then $(MAKE) -f metric.mk _ref/libfslic_ref_metric.so; else echo "no $(REF): keeping prebuilt _ref"; fi

_ref/libfslic_ref.so:
	$(MAKE) -f Makefile ref

_ref/libfslic_ref_metric.so: ref_shim_metric.cpp _ref/libfslic_ref.so
	$(CXX) $(REF_FLAGS) -I$(REF)/src -shared ref_shim_metric.cpp -o _ref/libfslic_ref_metric.so \
		-L_ref -lfslic_ref -Wl,-rpath,'$$ORIGIN'

clean:
	rm -f liboracle_metric.so _ref/libfslic_ref_metric.so
