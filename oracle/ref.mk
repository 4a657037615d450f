# oracle/_ref: the reference's OWN discrete-BIC sources, compiled where they lie in an urlearning-cpp checkout (REF, by
# default $URLEARNING_CPP_SRC: the directory that holds urlearning/) against the shim headers in oracle/shim/ (Boost is absent).  Only ref_driver.cpp is ours.  Output: oracle/_ref/libref_bic.so
# (git-ignored, travels to the GPU box).  Reference sources are never copied into the repo.
REF ?= $(URLEARNING_CPP_SRC)
ifeq ($(strip $(REF)),)
$(error set REF or URLEARNING_CPP_SRC to an urlearning-cpp source checkout)
endif
CXX = $(shell test -x /usr/bin/g++ && echo /usr/bin/g++ || echo g++)
# the reference's own flags (urlearning/Jamroot:14-45): -std=c++11 -fno-strict-aliasing; -w: its warnings are not ours
CXXFLAGS = -std=c++11 -fno-strict-aliasing -O2 -fPIC -w -pthread -I shim -I $(REF)
SRC = base/bayesian_network.cpp base/skeleton.cpp ad_tree/ad_tree.cpp ad_tree/ad_node.cpp ad_tree/vary_node.cpp \
      scoring_function/log_likelihood_calculator.cpp scoring_function/bic_scoring_function.cpp scoring_function/score_calculator.cpp \
      scoring_function/fnml_scoring_function.cpp scoring_function/bdeu_scoring_function.cpp
# the search side (consumers of the .pss): the reader, the best-score structures, the static pattern database, the heap
SEARCH_SRC = score_cache/score_cache.cpp score_cache/sparse_parent_list.cpp score_cache/sparse_parent_bitwise.cpp score_cache/sparse_parent_tree.cpp \
      heuristic/static_pattern_database.cpp priority_queue/priority_queue.cpp base/bayesian_network.cpp base/skeleton.cpp
OUT = _ref
# the Triplet A* driver (astar/triplet_astar.cpp) as a binary: its main() is renamed away, ref_triplet_driver.cpp supplies one
TRIPLET_SRC = heuristic/static_pattern_database.cpp heuristic/dynamic_pattern_database.cpp heuristic/combined_pattern_database.cpp \
      heuristic/file_pattern_database.cpp priority_queue/priority_queue.cpp base/bayesian_network.cpp base/skeleton.cpp \
      score_cache/score_cache.cpp score_cache/sparse_parent_list.cpp score_cache/sparse_parent_bitwise.cpp score_cache/sparse_parent_tree.cpp
# the continuous-BIC scoring function (BIC_OLS.cpp) over a minimal Armadillo / mlpack (shim_arma/): pins the reference's own code
# around the regression, see ref_cbic_driver.cpp
CBIC_SRC = base/bayesian_network.cpp scoring_function/BIC_OLS.cpp scoring_function/score_calculator.cpp
# the `score` binary itself: the reference's score/score_main.cpp with its own main(), every scoring function of this project's
# path behind it (BIC, fNML, BDeu over its AD-tree; cBIC over shim_arma), Boost replaced by working shims (program_options
# parses, thread runs)
SCORE_SRC = score/score_main.cpp base/bayesian_network.cpp base/skeleton.cpp ad_tree/ad_tree.cpp ad_tree/ad_node.cpp ad_tree/vary_node.cpp \
      scoring_function/log_likelihood_calculator.cpp scoring_function/bic_scoring_function.cpp scoring_function/fnml_scoring_function.cpp \
      scoring_function/bdeu_scoring_function.cpp scoring_function/score_calculator.cpp scoring_function/BIC_OLS.cpp
all: $(OUT)/libref_bic.so $(OUT)/libref_search.so $(OUT)/ref_triplet $(OUT)/libref_cbic.so $(OUT)/ref_score
$(OUT)/ref_score: $(addprefix $(REF)/urlearning/,$(SCORE_SRC)) $(wildcard shim/boost/*.hpp) shim_arma/armadillo $(wildcard shim_arma/mlpack/*.hpp) $(wildcard shim_arma/urlearning/scoring_function/*.h)
	@mkdir -p $(OUT)
	$(CXX) -std=c++11 -fno-strict-aliasing -O2 -w -pthread -include set -include map -include fstream -I shim_arma -I shim -I $(REF) -o $@ $(addprefix $(REF)/urlearning/,$(SCORE_SRC))
$(OUT)/libref_cbic.so: ref_cbic_driver.cpp $(addprefix $(REF)/urlearning/,$(CBIC_SRC)) $(wildcard shim/boost/*.hpp) shim_arma/armadillo $(wildcard shim_arma/mlpack/*.hpp) $(wildcard shim_arma/mlpack/methods/linear_regression/*.hpp)
	@mkdir -p $(OUT)
	$(CXX) -std=c++11 -fno-strict-aliasing -O2 -fPIC -w -pthread -I shim_arma -I shim -I $(REF) -shared -Wl,-Bsymbolic -o $@ ref_cbic_driver.cpp $(addprefix $(REF)/urlearning/,$(CBIC_SRC))
$(OUT)/ref_triplet: ref_triplet_driver.cpp $(REF)/urlearning/astar/triplet_astar.cpp $(addprefix $(REF)/urlearning/,$(TRIPLET_SRC)) $(wildcard shim/boost/*.hpp) $(wildcard shim/boost/*/*.hpp)
	@mkdir -p $(OUT)
	$(CXX) -std=c++11 -fno-strict-aliasing -O1 -w -pthread -include set -include map -include fstream -I shim -I $(REF) -Dmain=ref_triplet_unused_main -c $(REF)/urlearning/astar/triplet_astar.cpp -o $(OUT)/triplet_astar.o
	$(CXX) -std=c++11 -fno-strict-aliasing -O1 -w -pthread -include set -include map -include fstream -I shim -I $(REF) -o $@ ref_triplet_driver.cpp $(OUT)/triplet_astar.o $(addprefix $(REF)/urlearning/,$(TRIPLET_SRC))
	@rm -f $(OUT)/triplet_astar.o
$(OUT)/libref_search.so: ref_search_driver.cpp $(addprefix $(REF)/urlearning/,$(SEARCH_SRC)) $(wildcard shim/boost/*.hpp)
	@mkdir -p $(OUT)
	$(CXX) $(CXXFLAGS) -shared -Wl,-Bsymbolic -o $@ ref_search_driver.cpp $(addprefix $(REF)/urlearning/,$(SEARCH_SRC))
$(OUT)/libref_bic.so: ref_driver.cpp $(addprefix $(REF)/urlearning/,$(SRC)) $(wildcard shim/boost/*.hpp)
	@mkdir -p $(OUT)
	$(CXX) $(CXXFLAGS) -shared -Wl,-Bsymbolic -o $@ ref_driver.cpp $(addprefix $(REF)/urlearning/,$(SRC))
