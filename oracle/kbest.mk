# Builds the k-best Viterbi CPU oracle (test infrastructure only; see kbest_oracle.h), with the flags of Makefile.
CC      := /usr/bin/gcc
CFLAGS  ?= -O2 -ffp-contract=off -fno-fast-math -fopenmp -fPIC -Wall -Wextra -std=c11

all: libkbest_oracle.so

libkbest_oracle.so: kbest_oracle.c kbest_oracle.h cv_oracle.h
	$(CC) $(CFLAGS) -shared kbest_oracle.c -o $@ -lm

clean:
	rm -f libkbest_oracle.so
