# Builds libcoxgraph_b200.so (sm_100a only) and the CPU oracle (test infrastructure).
NVCC ?= /usr/local/cuda/bin/nvcc
ARCH  = -gencode arch=compute_100a,code=sm_100a
# -fmad=false / -ffp-contract=off: no FMA contraction anywhere — every float op on the path is
# the plain IEEE single-precision one, which is what makes block allocation bit-exact.
# alpha byte of a default-constructed voxblox::Color (csrc/cg_math.cuh); pass the same value to
# the oracle (`make -C oracle DEFAULT_ALPHA=...`) when changing it
DEFAULT_ALPHA ?= 255
NVFLAGS = $(ARCH) -DCG_DEFAULT_ALPHA=$(DEFAULT_ALPHA) -O3 -std=c++17 -lineinfo -fmad=false -prec-div=true -prec-sqrt=true -ftz=false \
          -Xcompiler -fPIC,-ffp-contract=off,-fno-fast-math,-Wall -Iinclude --expt-relaxed-constexpr
SRC  = coxgraph_b200/csrc
OBJ  = build/obj
LIB  = coxgraph_b200/lib/libcoxgraph_b200.so
HDRS = $(SRC)/cg_math.cuh $(SRC)/cg_internal.cuh $(SRC)/host_stage.cuh $(SRC)/cg_raycast_direct.cuh \
       $(SRC)/integrate.cuh include/coxgraph_b200.h
OBJS = $(OBJ)/layer.o $(OBJ)/integrate.o $(OBJ)/integrate_front.o $(OBJ)/integrate_back.o $(OBJ)/integrate_depth.o $(OBJ)/merge.o $(OBJ)/exchange.o $(OBJ)/comm.o $(OBJ)/mesh_recover.o $(OBJ)/mesh.o $(OBJ)/mesh_connect.o $(OBJ)/esdf.o $(OBJ)/host_stage.o $(OBJ)/selftest.o

HOSTCHK = build/host_api_check
DEPTHCHK = build/depth_api_check
ESDFCHK = build/esdf_update_check

all: $(LIB) oracle $(HOSTCHK) $(DEPTHCHK) $(ESDFCHK)

$(OBJ)/%.o: $(SRC)/%.cu $(HDRS)
	@mkdir -p $(OBJ)
	$(NVCC) $(NVFLAGS) -c $< -o $@

$(LIB): $(OBJS)
	@mkdir -p coxgraph_b200/lib
	$(NVCC) $(ARCH) -shared -o $@ $(OBJS) -cudart static -ldl -lpthread

oracle:
	$(MAKE) -C oracle -s DEFAULT_ALPHA=$(DEFAULT_ALPHA)

# C++ host API driver (tests/test_host_cpp.py): plain g++, links only the C ABI
$(HOSTCHK): tests/host/host_api_check.cc coxgraph_b200/host/coxgraph_b200.hpp include/coxgraph_b200.h $(LIB)
	g++ -std=c++17 -O1 -Wall -Wextra tests/host/host_api_check.cc -o $@ -Lcoxgraph_b200/lib \
	    -lcoxgraph_b200 -Wl,-rpath,'$$ORIGIN/../coxgraph_b200/lib'

# C++ depth-image driver (tests/test_host_depth.py)
$(DEPTHCHK): tests/host/depth_api_check.cc coxgraph_b200/host/coxgraph_b200.hpp include/coxgraph_b200.h $(LIB)
	g++ -std=c++17 -O1 -Wall -Wextra tests/host/depth_api_check.cc -o $@ -Lcoxgraph_b200/lib \
	    -lcoxgraph_b200 -Wl,-rpath,'$$ORIGIN/../coxgraph_b200/lib'

# C++ incremental-ESDF driver (tests/test_host_esdf_update.py)
$(ESDFCHK): tests/host/esdf_update_check.cc coxgraph_b200/host/coxgraph_b200.hpp include/coxgraph_b200.h $(LIB)
	g++ -std=c++17 -O1 -Wall -Wextra tests/host/esdf_update_check.cc -o $@ -Lcoxgraph_b200/lib \
	    -lcoxgraph_b200 -Wl,-rpath,'$$ORIGIN/../coxgraph_b200/lib'

clean:
	rm -rf build coxgraph_b200/lib oracle/_build

.PHONY: all oracle clean
