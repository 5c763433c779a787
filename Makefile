# Builds the product: libsw4b200.so (CUDA kernels + host engine behind the C ABI) and the drop-in CLIs.
# sm_100a only; artefacts stay in-tree (git-ignored) so they travel to the GPU box.
NVCC     ?= nvcc
CXXHOST  := $(shell command -v /usr/bin/g++ || echo g++)
ARCH     := -gencode arch=compute_100a,code=sm_100a
NVFLAGS  := -std=c++17 -O3 -lineinfo $(ARCH) -ccbin $(CXXHOST) -Xcompiler -fPIC,-Wall,-Wno-unused-function -Xptxas -v
CSRC     := cudasw4_b200/csrc
LIB      := cudasw4_b200/libsw4b200.so
HDRS     := $(wildcard $(CSRC)/*.cuh $(CSRC)/*.hpp) include/sw4b200.h

.PHONY: all lib cli oracle clean variant
all: lib cli

# one object per kernel family so that they build in parallel (make -j) and independently of the host engine
# (the two-row kernel additionally once per gap-score set whose values are compiled in as immediates, -DSW4_GAPS=n)
UNITS    := engine launch_s16 launch_s16_g1 launch_s16_g2 launch_s16_g3 launch_s16_multi launch_s16_multi_g1 launch_s16_multi_g2 launch_s16_multi_g3 launch_s16_wide launch_long launch_coords
OBJS     := $(patsubst %,build/%.o,$(UNITS))

lib: $(LIB)
build/launch_s16_g%.o: $(CSRC)/launch_s16.cu $(HDRS)
	@mkdir -p build
	$(NVCC) $(NVFLAGS) -DSW4_GAPS=$* -c -o $@ $< 2> build/launch_s16_g$*.ptxas.log || (cat build/launch_s16_g$*.ptxas.log; exit 1)
build/launch_s16_multi_g%.o: $(CSRC)/launch_s16_multi.cu $(HDRS)
	@mkdir -p build
	$(NVCC) $(NVFLAGS) -DSW4_GAPS=$* -c -o $@ $< 2> build/launch_s16_multi_g$*.ptxas.log || (cat build/launch_s16_multi_g$*.ptxas.log; exit 1)
build/%.o: $(CSRC)/%.cu $(HDRS)
	@mkdir -p build
	$(NVCC) $(NVFLAGS) -c -o $@ $< 2> build/$*.ptxas.log || (cat build/$*.ptxas.log; exit 1)
$(LIB): $(OBJS)
	$(NVCC) $(ARCH) -shared -o $@ $(OBJS) -lpthread
	@cat $(patsubst %,build/%.ptxas.log,$(UNITS)) > build/engine.ptxas.log
	@grep -E "error|spill" build/engine.ptxas.log | grep -v " 0 bytes spill stores, 0 bytes spill loads" | sort | uniq -c | sort -rn | head -20 || true

# kernel-variant sweeps (development aid): make variant NAME=x DEFS="-DSW4_..."  ->  build/variants/x.so
variant:
	@mkdir -p build/variants/$(NAME)
	@for u in $(UNITS); do src=$$(echo $$u | sed -E 's/_g[0-9]+$$//'); g=$$(echo $$u | sed -nE 's/.*_g([0-9]+)$$/-DSW4_GAPS=\1/p'); echo "$(NVCC) $(NVFLAGS) $(DEFS) $$g -c -o build/variants/$(NAME)/$$u.o $(CSRC)/$$src.cu 2> build/variants/$(NAME)/$$u.ptxas.log"; done | xargs -P 8 -I{} sh -c "{}"
	$(NVCC) $(ARCH) -shared -o build/variants/$(NAME).so $(patsubst %,build/variants/$(NAME)/%.o,$(UNITS)) -lpthread
	@cat build/variants/$(NAME)/*.ptxas.log | grep -E "spill" | grep -v " 0 bytes spill stores, 0 bytes spill loads" | sort | uniq -c | sort -rn | head -8 || true

cli: build/align build/makedb
build/align: $(CSRC)/cli_align.cpp include/cudasw4.cuh include/sw4b200.h $(CSRC)/fasta_reader.hpp $(CSRC)/blosum_tables.hpp $(LIB)
	@mkdir -p build
	$(CXXHOST) -std=c++17 -O2 -Wall -Iinclude -o $@ $(CSRC)/cli_align.cpp -Lcudasw4_b200 -lsw4b200 -Wl,-rpath,'$$ORIGIN/../cudasw4_b200' -lz
build/makedb: $(CSRC)/cli_makedb.cpp $(CSRC)/fasta_reader.hpp
	@mkdir -p build
	$(CXXHOST) -std=c++17 -O2 -Wall -o $@ $(CSRC)/cli_makedb.cpp -lz

oracle:
	$(MAKE) -C oracle all

clean:
	rm -f $(LIB) build/align build/makedb build/*.log build/*.o
