# oracle/apps.mk — the CPU oracle of the apps beyond the seven pipelines of oracle/Makefile (harris, unsharp), and, when
# the reference is present, their unmodified harnesses and RunGen drivers linked against libhalide_b200.so into
# oracle/_ref (compiled from where they lie, never copied).  Same flags as oracle/Makefile.
#     make -C oracle -f apps.mk
CXX = /usr/bin/g++
CXXFLAGS = -O3 -mavx2 -fPIC -std=c++17 -fopenmp -ffp-contract=off -fno-fast-math -Wall -Wno-unknown-pragmas
REF ?= /root/reference
APPS_SRCS = oracle_harris.cpp oracle_unsharp.cpp

all: liboracle_apps.so ref_apps

liboracle_apps.so: $(APPS_SRCS) oracle_apps.h oracle.h halide_math.h
	$(CXX) $(CXXFLAGS) -shared -o $@ $(APPS_SRCS)

# apps/<app>/filter.cpp calls <app>(input, output) and <app>_auto_schedule(...) from include/<app>.h and
# include/<app>_auto_schedule.h; tools/RunGenMain.cpp + halide_b200/registration/<app>_registration.cpp is the generic
# benchmark driver.  Both need ../halide_b200/libhalide_b200.so built first.
ref_apps:
	@if [ -d $(REF)/apps/harris ] && [ -d $(REF)/apps/unsharp ]; then \
	  mkdir -p _ref; \
	  for app in harris unsharp; do \
	    $(CXX) -O2 -std=c++17 -I../include -I$(REF)/src/runtime -I$(REF)/tools -DHALIDE_NO_PNG -DHALIDE_NO_JPEG \
	       $(REF)/apps/$$app/filter.cpp -o _ref/$${app}_filter -L../halide_b200 -lhalide_b200 \
	       -Wl,-rpath,'$$ORIGIN/../../halide_b200' -lpthread -ldl && \
	    echo "built oracle/_ref/$${app}_filter (reference harness apps/$$app/filter.cpp, unmodified, linked against libhalide_b200.so)"; \
	    $(CXX) -O2 -std=c++17 -I../include -I$(REF)/src/runtime -I$(REF)/tools -DHALIDE_NO_PNG -DHALIDE_NO_JPEG \
	       $(REF)/tools/RunGenMain.cpp ../halide_b200/registration/$${app}_registration.cpp -o _ref/$${app}_rungen \
	       -L../halide_b200 -lhalide_b200 -Wl,-rpath,'$$ORIGIN/../../halide_b200' -lpthread -ldl && \
	    echo "built oracle/_ref/$${app}_rungen (reference tools/RunGenMain.cpp, unmodified, + our registration TU)"; \
	  done; \
	else echo "reference not present: keeping prebuilt oracle/_ref harris / unsharp binaries"; fi

clean:
	rm -f liboracle_apps.so
.PHONY: all ref_apps clean
