# oracle/seam2_strand.mk — TEST INFRASTRUCTURE ONLY: the seam-2 cluster driver with --strand selectable.
#
#   make -C oracle -f Makefile -f seam2_strand.mk strand
#
# Reuses oracle/Makefile's objects and variables.  _ref/seam2_cluster_driver_strand_{ref,gpu} are the unchanged
# seam2_cluster_driver.cpp linked as in oracle/Makefile, plus seam2_strand_wrap.cpp, which sets opt_strand from
# SEAM2_STRAND=both|plus before cluster_session_init runs.
CSI_SYM := _Z20cluster_session_initP17cluster_session_sRK10ParametersR7DbindexRK8Database

.PHONY: strand
ifneq ($(wildcard $(SRC)/vsearch.cc),)
strand: $(OUT)/seam2_cluster_driver_strand_ref $(OUT)/seam2_cluster_driver_strand_gpu
else
strand:
	@echo "reference sources not present at $(SRC): using prebuilt $(OUT)/ if any"
endif

$(OBJ)/seam2_strand_wrap.o: seam2_strand_wrap.cpp
	@mkdir -p $(dir $@)
	$(CXX) $(CXXFL) -c $< -o $@
$(OUT)/seam2_cluster_driver_strand_ref: seam2_cluster_driver.cpp $(OBJ)/seam2_strand_wrap.o $(OUT)/libvsearch_ref.a
	$(CXX) $(CXXFL) -o $@ $< $(OBJ)/seam2_strand_wrap.o $(OUT)/libvsearch_ref.a -Wl,--wrap=$(CSI_SYM) -lpthread -ldl
$(OUT)/seam2_cluster_driver_strand_gpu: seam2_cluster_driver.cpp $(OBJ)/seam2_strand_wrap.o $(SEAM2C_OBJS) $(VSG_DIR)/libvsg.so
	$(CXX) $(CXXFL) -o $@ $< $(OBJ)/seam2_strand_wrap.o $(SEAM2C_OBJS) -L$(VSG_DIR) -lvsg -Wl,-rpath,'$$ORIGIN/../../vsearch_b200/csrc' \
	    -Wl,--wrap=$(CSI_SYM) -lpthread -ldl
