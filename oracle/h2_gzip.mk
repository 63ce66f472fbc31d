# Builds oracle/liboracle_h2gzip.so (test infrastructure): orc_h2_decompress on top of liboracle.so.  `make -f oracle/h2_gzip.mk`
CC ?= gcc
HERE := $(dir $(abspath $(lastword $(MAKEFILE_LIST))))

all: $(HERE)liboracle_h2gzip.so

$(HERE)liboracle_h2gzip.so: $(HERE)b2_oracle_h2_gzip.c $(HERE)b2_oracle_h2_gzip.h $(HERE)b2_oracle.h $(HERE)../include/b2rpc.h $(HERE)liboracle.so
	$(CC) -O2 -g -std=c11 -D_GNU_SOURCE -fPIC -shared -Wall -Wextra -o $@ $(HERE)b2_oracle_h2_gzip.c -L$(HERE) -loracle -Wl,-rpath,$(HERE)

$(HERE)liboracle.so:
	$(MAKE) -C $(HERE)

clean:
	rm -f $(HERE)liboracle_h2gzip.so
.PHONY: all clean
