# oracle/polya.mk — TEST INFRASTRUCTURE ONLY: the checkers of `nanopolish polya` (section 8f N5), on top of oracle/Makefile
# (its compiler, flags, include paths, reference objects and their rules are used as they are).
#   make -C oracle -f polya.mk polya-port   oracle/libnpo_polya.so         plain-C restatement (np_polya.c)
#   make -C oracle -f polya.mk polya-ref    oracle/_ref/libnpref_polya.so  the reference's src/nanopolish_polya_estimator.cpp
#                                           compiled inside ref_polya_harness.cpp and linked with the same reference objects as
#                                           libnpref.so under --gc-sections (only where $(REF) exists; elsewhere the prebuilt one)
include Makefile
.DEFAULT_GOAL := polya-port
.PHONY: polya-port polya-ref

polya-port: libnpo_polya.so

libnpo_polya.so: np_polya.c
	$(CC) -O2 -std=c99 -fPIC -shared -fopenmp -ffp-contract=off -o $@ np_polya.c -lm

ifneq ($(wildcard $(REF)/src/nanopolish_polya_estimator.cpp),)
polya-ref: $(OUT)/libnpref_polya.so
else
polya-ref:
	@echo "oracle/polya.mk: $(REF) not present: using prebuilt $(OUT)/libnpref_polya.so if any"
endif

# the harness TU includes ref_harness.cpp (the reads it builds) and the reference's polya .cpp; one section per function, as for
# the other CLI translation units, so that --gc-sections drops the CLI code
$(OUT)/obj/ref_polya_harness.o: REFFLAGS += -ffunction-sections -fdata-sections
$(OUT)/obj/ref_polya_harness.o: ref_polya_harness.cpp ref_harness.cpp shim/Eigen/Dense $(REF)/src/nanopolish_polya_estimator.cpp
	@mkdir -p $(OUT)/obj
	$(CXX) $(REFFLAGS) $(REFINC) -c $< -o $@

$(OUT)/libnpref_polya.so: $(REF_OBJS) $(REF_GC_OBJS) $(OUT)/obj/ref_polya_harness.o npref.map
	$(CXX) -shared -fopenmp -Wl,--gc-sections -Wl,--version-script=npref.map -o $@ $(REF_OBJS) $(REF_GC_OBJS) $(OUT)/obj/ref_polya_harness.o
