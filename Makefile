# Builds libocmps.so (sm_100a only) in-tree.
NVCC ?= nvcc
ARCH := -gencode arch=compute_100a,code=sm_100a
NVFLAGS := $(ARCH) -O3 -lineinfo -std=c++17 -Xcompiler -fPIC -Xptxas -v
SRC := optimalcontrolmps_b200/csrc
OBJS := $(SRC)/zgemm.o $(SRC)/decomp.o $(SRC)/elementwise.o $(SRC)/dmrg.o $(SRC)/engine.o
LIB := optimalcontrolmps_b200/libocmps.so

all: $(LIB)

$(SRC)/%.o: $(SRC)/%.cu $(SRC)/ocmps_internal.h include/ocmps.h
	$(NVCC) $(NVFLAGS) -c $< -o $@

$(LIB): $(OBJS)
	$(NVCC) $(ARCH) -shared -o $@ $(OBJS) -lcudart

clean:
	rm -f $(OBJS) $(LIB)
