# TEST INFRASTRUCTURE -- the reference producer with its almanac enabled (ref_harness/ref_dump_alm.c, switch
# --almanac: the reference then reads almanac.sem from its working directory). Nothing here is product code.
#
#   make -C oracle -f alm.mk   -> oracle/_ref/ref_dump{12,32}_alm, ref_dump12_u32_alm  (only when $(REF) exists)
# Same flags as Makefile / u32.mk; the _u32 binary force-includes a temporary copy of the reference's gps.h without
# `#define FLOAT_CARR_PHASE`, as u32.mk does. The reference sources are compiled where they lie.
REF      ?= /root/reference
OUT      := _ref
H        := ref_harness
CC       ?= gcc
STD      := -std=c11 -D_GNU_SOURCE -ffp-contract=off
SHIPPED  := $(STD) -Og -g
INC      := -I$(H) -I$(REF)
LIBS     := -lm -lpthread -lz
W        := -w
SRCS     := $(H)/ref_dump_alm.c $(H)/ref_dump.c $(H)/gui_stub.c

REF_BINS := $(OUT)/ref_dump12_alm $(OUT)/ref_dump32_alm $(OUT)/ref_dump12_u32_alm

all: $(if $(wildcard $(REF)/gps.c),$(REF_BINS),)

$(OUT):
	mkdir -p $(OUT)

$(OUT)/ref_dump12_alm: $(SRCS) | $(OUT)
	$(CC) $(SHIPPED) $(W) $(INC) -DORACLE_DUMP_PARAMS -o $@ $(H)/ref_dump_alm.c $(H)/gui_stub.c $(REF)/almanac.c $(LIBS)
$(OUT)/ref_dump32_alm: $(SRCS) | $(OUT)
	$(CC) $(SHIPPED) $(W) $(INC) -DORACLE_DUMP_PARAMS -DORACLE_MAX_CHAN=32 -o $@ $(H)/ref_dump_alm.c $(H)/gui_stub.c \
	    $(REF)/almanac.c $(LIBS)

u32_hdr = grep -qx '\#define FLOAT_CARR_PHASE' $(REF)/gps.h && grep -vx '\#define FLOAT_CARR_PHASE' $(REF)/gps.h > $(1)/gps.h

$(OUT)/ref_dump12_u32_alm: $(SRCS) | $(OUT)
	T=$$(mktemp -d) && $(call u32_hdr,$$T) && \
	$(CC) $(SHIPPED) $(W) -include $$T/gps.h -I$$T $(INC) -DORACLE_DUMP_PARAMS -o $@ $(H)/ref_dump_alm.c $(H)/gui_stub.c \
	    $(REF)/almanac.c $(LIBS); rc=$$?; rm -rf $$T; exit $$rc

.PHONY: all
