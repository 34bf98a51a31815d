# TEST-ONLY: builds the check program of the key slots of act::Engine and its keyed overload (include/act.hpp) against the product
# library (no GPU needed to compile and link).  usage: make -C tests/cpp -f keys_hpp_check.mk
PKG := ../../anonymous-credit-tokens_b200
keys_hpp_check: keys_hpp_check.cpp ../../include/act.hpp ../../include/act_engine.h $(PKG)/libact_b200.so
	g++ -std=c++17 -O1 -Wall -Wextra -I ../../include -o $@ keys_hpp_check.cpp -L $(PKG) -lact_b200 -Wl,-rpath,'$$ORIGIN/$(PKG)'
clean:
	rm -f keys_hpp_check
