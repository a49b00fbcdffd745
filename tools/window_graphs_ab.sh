for W in 3 10; do for G in 4 8 16; do python tools/window_bench.py --W $W --graphs $G --nonterm --eps $( [ $W = 3 ] && echo 0.30 || echo 0.45 ); done; done
