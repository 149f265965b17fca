# TEST INFRASTRUCTURE -- the reference's INTEGER carrier build (gps.h:17 `#define FLOAT_CARR_PHASE` absent) and the
# oracle of that build. Nothing here is product code.
#
#   make -C oracle -f u32.mk   -> oracle/_ref/liboracle_gpsl1_u32.so (C restatement, always)
#                                 oracle/_ref/ref_*_u32            (the reference itself, only when $(REF) exists)
# Every recipe writes a TEMPORARY copy of the reference's gps.h without the line `#define FLOAT_CARR_PHASE` (checked
# by content: the recipe fails when the line is absent) and force-includes it ahead of everything, so that every
# later `#include "gps.h"` of the reference's sources hits its include guard. The copy never enters the repository;
# the reference sources are compiled where they lie, as in Makefile.
REF      ?= /root/reference
OUT      := _ref
H        := ref_harness
CC       ?= gcc
STD      := -std=c11 -D_GNU_SOURCE -ffp-contract=off
SHIPPED  := $(STD) -Og -g
FAST     := $(STD) -O2 -fstack-reuse=none
INC      := -I$(H) -I$(REF)
LIBS     := -lm -lpthread -lz
W        := -w
GPSLIB   := ../multi-sdr-gps-sim_b200
RPATH    := -Wl,-rpath,'$$ORIGIN/../../multi-sdr-gps-sim_b200'

REF_BINS := $(OUT)/ref_dump12_u32 $(OUT)/ref_dump32_u32 $(OUT)/ref_run32_u32_fast
DROPIN   := $(OUT)/ref_gpsb200_12_u32

all: $(OUT)/liboracle_gpsl1_u32.so $(if $(wildcard $(REF)/gps.c),$(REF_BINS) $(if $(wildcard $(GPSLIB)/libgpsb200.so),$(DROPIN),),)

$(OUT):
	mkdir -p $(OUT)

$(OUT)/liboracle_gpsl1_u32.so: gpsl1_oracle.c gpsl1_oracle_u32.c gpsl1_oracle.h | $(OUT)
	$(CC) $(STD) -O2 -fPIC -shared -o $@ gpsl1_oracle.c gpsl1_oracle_u32.c -lm

# $(call u32_hdr,DIR): DIR/gps.h = the reference's gps.h without `#define FLOAT_CARR_PHASE`
u32_hdr = grep -qx '\#define FLOAT_CARR_PHASE' $(REF)/gps.h && grep -vx '\#define FLOAT_CARR_PHASE' $(REF)/gps.h > $(1)/gps.h

$(OUT)/ref_dump12_u32: $(H)/ref_dump.c $(H)/gui_stub.c | $(OUT)
	T=$$(mktemp -d) && $(call u32_hdr,$$T) && \
	$(CC) $(SHIPPED) $(W) -include $$T/gps.h -I$$T $(INC) -DORACLE_DUMP_PARAMS -o $@ $(H)/ref_dump.c $(H)/gui_stub.c \
	    $(REF)/almanac.c $(LIBS); rc=$$?; rm -rf $$T; exit $$rc
$(OUT)/ref_dump32_u32: $(H)/ref_dump.c $(H)/gui_stub.c | $(OUT)
	T=$$(mktemp -d) && $(call u32_hdr,$$T) && \
	$(CC) $(SHIPPED) $(W) -include $$T/gps.h -I$$T $(INC) -DORACLE_DUMP_PARAMS -DORACLE_MAX_CHAN=32 -o $@ $(H)/ref_dump.c \
	    $(H)/gui_stub.c $(REF)/almanac.c $(LIBS); rc=$$?; rm -rf $$T; exit $$rc
$(OUT)/ref_run32_u32_fast: $(H)/ref_dump.c $(H)/gui_stub.c | $(OUT)
	T=$$(mktemp -d) && $(call u32_hdr,$$T) && \
	$(CC) $(FAST) $(W) -include $$T/gps.h -I$$T $(INC) -DORACLE_MAX_CHAN=32 -o $@ $(H)/ref_dump.c $(H)/gui_stub.c \
	    $(REF)/almanac.c $(LIBS); rc=$$?; rm -rf $$T; exit $$rc

# the drop-in program (Makefile: ref_gpsb200_12) built on the integer carrier: the temporary gps.h and the setup
# snippet that selects GPSB200_CARRIER_U32 sit next to the temporary gps.c, where its quoted includes look first
$(OUT)/ref_gpsb200_12_u32: $(H)/apply_integration.py $(H)/integration_decl.inc $(H)/integration_setup_u32.inc \
        $(H)/integration_block.inc $(H)/integration_teardown.inc $(H)/ref_stock_main.c $(H)/gui_stub.c \
        $(GPSLIB)/libgpsb200.so | $(OUT)
	T=$$(mktemp -d) && $(call u32_hdr,$$T) && cp $(H)/integration_setup_u32.inc $$T/integration_setup.inc && \
	python3 $(H)/apply_integration.py $(REF)/gps.c $$T/gps_gpsb200.c && \
	$(CC) $(SHIPPED) $(W) -include $$T/gps.h -I$$T $(INC) -I../include -o $@ $(H)/ref_stock_main.c $(H)/gui_stub.c \
	    $$T/gps_gpsb200.c $(REF)/sdr.c $(REF)/sdr_iqfile.c $(REF)/almanac.c -L$(GPSLIB) -lgpsb200 $(RPATH) $(LIBS); \
	rc=$$?; rm -rf $$T; exit $$rc

.PHONY: all
