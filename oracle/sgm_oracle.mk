# TEST INFRASTRUCTURE.  Builds oracle/_build/libsgmoracle.so, the plain-C restatement of the semi-global matching of
# visocu_disparity (sgm_oracle.c), loaded by sgm_oracle.py.  make -C oracle -f sgm_oracle.mk
HERE := $(dir $(abspath $(lastword $(MAKEFILE_LIST))))
CC ?= gcc
MARCH ?= x86-64-v3

all: $(HERE)_build/libsgmoracle.so
$(HERE)_build/libsgmoracle.so: $(HERE)sgm_oracle.c $(HERE)sgm_oracle.h
	@mkdir -p $(HERE)_build
	$(CC) -std=c11 -O2 -march=$(MARCH) -fPIC -shared -Wall -Wextra -o $@ $(HERE)sgm_oracle.c

clean:
	rm -f $(HERE)_build/libsgmoracle.so
.PHONY: all clean
