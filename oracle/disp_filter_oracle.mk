# TEST INFRASTRUCTURE.  Builds oracle/_build/libdispfilteroracle.so, the plain-C restatement of the disparity
# post-filters (disp_filter_oracle.c), loaded by disp_filter_oracle.py.  make -C oracle -f disp_filter_oracle.mk
HERE := $(dir $(abspath $(lastword $(MAKEFILE_LIST))))
CC ?= gcc
MARCH ?= x86-64-v3

all: $(HERE)_build/libdispfilteroracle.so
$(HERE)_build/libdispfilteroracle.so: $(HERE)disp_filter_oracle.c $(HERE)disp_filter_oracle.h
	@mkdir -p $(HERE)_build
	$(CC) -std=c11 -O2 -march=$(MARCH) -fPIC -shared -Wall -Wextra -o $@ $(HERE)disp_filter_oracle.c

clean:
	rm -f $(HERE)_build/libdispfilteroracle.so
.PHONY: all clean
