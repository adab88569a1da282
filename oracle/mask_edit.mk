# Builds the CPU restatement of the 3-D mask editor (test infrastructure; never linked into the
# product) as its own library beside liboracle.so.
# -ffp-contract=off: the reference (Rust) never fuses multiply-add.
CC ?= gcc
CFLAGS = -O2 -fPIC -shared -std=c11 -ffp-contract=off -fno-fast-math -Wall -Wno-unused-function

all: libmask_edit.so

libmask_edit.so: mask_edit.c
	$(CC) $(CFLAGS) -o $@ mask_edit.c -lm

clean:
	rm -f libmask_edit.so
