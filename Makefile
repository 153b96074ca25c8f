# zultra-b200 build: CUDA pipeline + C host library -> zultra_b200/libzultra_b200.so, CLI -> zultra_b200/zultra
NVCC ?= nvcc
CC ?= gcc
ARCH = -gencode arch=compute_100a,code=sm_100a
NVFLAGS = $(ARCH) -lineinfo -O3 -std=c++17 --extended-lambda -Xcompiler -fPIC -diag-suppress 177,550
CFLAGS = -O2 -fPIC -Wall -Iinclude
CS = zultra_b200/csrc
B = build

all: zultra_b200/libzultra_b200.so zultra_b200/zultra

$(B)/%.o: $(CS)/%.cu $(CS)/zb_core.h $(CS)/zb_rt.h $(CS)/zb_pipeline.h $(CS)/zb_engine.h include/zultra_cuda.h include/libzultra.h
	@mkdir -p $(B)
	$(NVCC) $(NVFLAGS) -c $< -o $@

$(B)/%.o: $(CS)/host/%.c include/libzultra.h include/zultra_cuda.h
	@mkdir -p $(B)
	$(CC) $(CFLAGS) -c $< -o $@

zultra_b200/libzultra_b200.so: $(B)/zb_capi.o $(B)/zb_prims.o $(B)/libzultra.o $(B)/frame.o $(B)/dictionary.o
	$(NVCC) $(ARCH) -shared -o $@ $^ -cudart static

zultra_b200/zultra: $(B)/zultra_cli.o zultra_b200/libzultra_b200.so
	$(CC) -o $@ $(B)/zultra_cli.o -Lzultra_b200 -lzultra_b200 -lz -Wl,-rpath,'$$ORIGIN'

emu:
	g++ -O2 -g -DZB_EMU -std=c++17 -fPIC -shared -I$(CS) -o tests/emu/libzb_emu.so tests/emu/zb_emu.cpp tests/emu/zb_batch_dict_emu.cpp tests/emu/zb_prims_emu.cpp

oracle:
	$(MAKE) -C oracle all

clean:
	rm -rf $(B) zultra_b200/libzultra_b200.so zultra_b200/zultra tests/emu/libzb_emu.so
.PHONY: all emu oracle clean
