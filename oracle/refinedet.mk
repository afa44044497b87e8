# oracle/refinedet.mk -- RefineDet test infrastructure (make -C oracle -f refinedet.mk)
#   liboracle_refinedet.so   plain-C fp64 restatement of refinedet/refinedet.cpp:553-790
#   _ref/libref_refinedet.so the REFERENCE's own PriorBox / decode / nms (refinedet.cpp, from `torch::Tensor PriorBox()`
#                            up to `void doInference`), extracted by pattern into _ref/ and compiled against the tensor
#                            library's C++ headers next to ref_wrap_refinedet.cpp.  Only where the reference tree exists;
#                            the extract never leaves _ref/ (git-ignored).
CC      ?= gcc
CXX     ?= g++
PYTHON  ?= python3
REF     ?= /root/reference
HERE    := $(dir $(abspath $(lastword $(MAKEFILE_LIST))))
CFLAGS  := -O2 -fPIC -shared -ffp-contract=off -fvisibility=hidden -Wall -Wextra -std=c11 -D_GNU_SOURCE
REFCPP  := $(REF)/refinedet/refinedet.cpp

all: $(HERE)liboracle_refinedet.so ref

$(HERE)liboracle_refinedet.so: $(HERE)refinedet_oracle.c
	$(CC) $(CFLAGS) -o $@ $< -lm

ifneq ($(wildcard $(REFCPP)),)
TORCH   := $(shell $(PYTHON) -c 'import torch, os; print(os.path.dirname(torch.__file__))')
CXXABI  := $(shell $(PYTHON) -c 'import torch; print(int(torch._C._GLIBCXX_USE_CXX11_ABI))')
CUDAINC := $(dir $(shell which nvcc 2>/dev/null || echo /usr/local/cuda/bin/nvcc))../include
# the reference's CMakeLists ends its flags with -O2 (after -Ofast, which it therefore overrides): IEEE arithmetic
REFFLAGS := -O2 -std=c++17 -fPIC -shared -w -fvisibility=hidden -D_GLIBCXX_USE_CXX11_ABI=$(CXXABI) \
            -I$(HERE)_ref -I$(TORCH)/include -I$(TORCH)/include/torch/csrc/api/include -I$(CUDAINC)
REFLIBS  := -L$(TORCH)/lib -Wl,--no-as-needed -ltorch -ltorch_cpu -ltorch_cuda -lc10 -lc10_cuda -Wl,-rpath,$(TORCH)/lib

ref: $(HERE)_ref/libref_refinedet.so

$(HERE)_ref/refinedet_postprocess.inc: $(REFCPP)
	@mkdir -p $(HERE)_ref
	awk '/^torch::Tensor PriorBox\(\)/{on=1} /^void doInference/{on=0} on' $< > $@
	@test -s $@ || (echo "PriorBox ... nms not found in $<" && rm -f $@ && false)

$(HERE)_ref/libref_refinedet.so: $(HERE)ref_wrap_refinedet.cpp $(HERE)_ref/refinedet_postprocess.inc
	$(CXX) $(REFFLAGS) -o $@ $< $(REFLIBS)
else
ref:
	@echo "reference tree not present: keeping prebuilt oracle/_ref/libref_refinedet.so"
endif

clean:
	rm -f $(HERE)liboracle_refinedet.so $(HERE)_ref/libref_refinedet.so $(HERE)_ref/refinedet_postprocess.inc
.PHONY: all ref clean
