# Builds the C-ABI library (sm_100a only), the C oracle pieces and, when the reference checkout is
# present, the reference oracle binary and the resql-b200 host front end.
NVCC ?= nvcc
NVCCFLAGS = -gencode arch=compute_100a,code=sm_100a -lineinfo -O3 -std=c++17 -Xcompiler -fPIC
CSRC = resql_b200/csrc
LIB = resql_b200/libresql_b200.so

all: $(LIB)

# The headers of the scan kernel as text, for run-time specializations (jit.h): each under the name its
# #include uses, so a specialization compiles exactly the source the library was built from.
JIT_HEADERS = include/resql_b200.h $(CSRC)/rq_internal.h $(CSRC)/device_util.cuh $(CSRC)/hash_kernels.cuh $(CSRC)/scan_kernel.cuh
JIT_INC = $(CSRC)/jit_sources.inc
$(JIT_INC): $(JIT_HEADERS)
	{ printf 'static const char* const kJitHeaderName[] = {'; \
	  for f in $^; do case $$f in include/*) printf '"../../%s", ' $$f;; *) printf '"%s", ' $${f##*/};; esac; done; \
	  printf '};\nstatic const char* const kJitHeaderText[] = {\n'; \
	  for f in $^; do printf 'R"rq_src('; cat $$f; printf ')rq_src",\n'; done; printf '};\n'; } > $@

$(LIB): $(CSRC)/engine.cu $(CSRC)/engine_exec.inl $(CSRC)/scan_kernel.cuh $(CSRC)/device_util.cuh $(CSRC)/hash_kernels.cuh \
        $(CSRC)/sort_kernels.cuh $(CSRC)/exchange_kernels.cuh $(CSRC)/host_narrow.h $(CSRC)/rq_internal.h $(CSRC)/dist.h include/resql_b200.h \
        $(CSRC)/jit.h $(JIT_INC)
	$(NVCC) $(NVCCFLAGS) -shared -o $@ $(CSRC)/engine.cu -ldl

ptxas-info: $(JIT_INC)
	$(NVCC) $(NVCCFLAGS) -Xptxas -v -shared -o /tmp/rq_ptxas.so $(CSRC)/engine.cu -ldl

oracle-ref:
	bash oracle/ref_build/build_ref.sh

host: $(LIB)
	bash resql_b200/host/build_host.sh

clean:
	rm -f $(LIB) $(JIT_INC) resql_b200/host/resql-b200

.PHONY: all ptxas-info oracle-ref host clean
