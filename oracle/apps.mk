# oracle/apps.mk — the CPU oracle of the apps beyond the seven pipelines of liboracle.so (harris, unsharp).  Their
# harnesses and RunGen drivers are built by oracle/Makefile's `ref` target.  Same flags as oracle/Makefile.
#     make -C oracle -f apps.mk
CXX = /usr/bin/g++
CXXFLAGS = -O3 -mavx2 -fPIC -std=c++17 -fopenmp -ffp-contract=off -fno-fast-math -Wall -Wno-unknown-pragmas
APPS_SRCS = oracle_harris.cpp oracle_unsharp.cpp

all: liboracle_apps.so

liboracle_apps.so: $(APPS_SRCS) oracle_apps.h oracle.h halide_math.h
	$(CXX) $(CXXFLAGS) -shared -o $@ $(APPS_SRCS)

clean:
	rm -f liboracle_apps.so
.PHONY: all clean
