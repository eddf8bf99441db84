# Builds the forward-backward CPU oracle (test infrastructure only; see fb_oracle.h), with the flags of Makefile.
CC      := /usr/bin/gcc
CFLAGS  ?= -O2 -ffp-contract=off -fno-fast-math -fopenmp -fPIC -Wall -Wextra -std=c11

all: libfb_oracle.so

libfb_oracle.so: fb_oracle.c fb_oracle.h cv_oracle.h
	$(CC) $(CFLAGS) -shared fb_oracle.c -o $@ -lm

clean:
	rm -f libfb_oracle.so
