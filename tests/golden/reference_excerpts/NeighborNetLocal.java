		this.additive = additive;
		myRandom = ThreadLocalRandom.current();
		rowPermutation = new int[numTaxa];
