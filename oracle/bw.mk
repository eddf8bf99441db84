# Builds the Baum-Welch CPU oracle (test infrastructure only; see bw_oracle.h), with the flags of Makefile.
CC      := /usr/bin/gcc
CFLAGS  ?= -O2 -ffp-contract=off -fno-fast-math -fopenmp -fPIC -Wall -Wextra -std=c11

all: libbw_oracle.so

libbw_oracle.so: bw_oracle.c bw_oracle.h cv_oracle.h
	$(CC) $(CFLAGS) -shared bw_oracle.c -o $@ -lm

clean:
	rm -f libbw_oracle.so
